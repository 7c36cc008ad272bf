"""Rating prediction (--rank 0, MSE) on the device-resident epoch and data parallel, without a GPU: BaseRunner.fit's
batch schedule with the labels beside the batches (one process and as a rank of a data-parallel job), and the argument
checks of the global MSE divisor and of the staged labels."""
import ctypes

import pytest
import torch

from dccf_b200 import _lib, build
from dccf_b200.runners.BaseRunner import BaseRunner
from test_fit_schedule import _dev, _Recorder


class _LabelRecorder(_Recorder):
    """The recording stand-in of test_fit_schedule, taking the label epoch of a rating-prediction epoch."""

    def __init__(self, item_num=1000, dp=None):
        _Recorder.__init__(self, item_num, dp)
        self.labels, self.stepwise_labels = [], []

    def begin_resident_epoch(self, X_epoch, draws, dropout, Y_epoch=None):
        assert Y_epoch is not None and Y_epoch.dtype == torch.float32
        assert tuple(Y_epoch.shape) == tuple(X_epoch.shape[:2])
        step = _Recorder.begin_resident_epoch(self, X_epoch, draws, dropout)
        inner, state = step, {'k': 0}

        def labelled():
            self.labels.append(Y_epoch[state['k']].clone())
            state['k'] += 1
            return inner()
        labelled.remaining, labelled.first = inner.remaining, None
        return labelled

    def train_step(self, fd):
        self.stepwise_labels.append(fd['Y'].clone())
        return _Recorder.train_step(self, fd)


class _RatingDP(object):
    rank = 0

    def __init__(self, batches):
        self._b = batches

    def prepare_batches(self, data, batch_size, train):
        return [dict(b) for b in self._b]


def _label(k, P):
    """The labels of batch k: distinct per batch and per pair, so a misaligned copy shows."""
    return k + torch.arange(P, dtype=torch.float32) / 64


def _batches(n_full, ragged, P=8):
    out = [{'X': _dev(torch.full((P, 2), k, dtype=torch.int64)), 'Y': _label(k, P)} for k in range(n_full)]
    if ragged:
        out.append({'X': _dev(torch.full((ragged, 2), n_full, dtype=torch.int64)), 'Y': _label(n_full, ragged)})
    return out


def _run(n_full, ragged, world, rank, monkeypatch):
    runner = BaseRunner(optimizer='Adam', learning_rate=1e-3, metrics='rmse', dropout=0.2)
    runner.show_progress = False
    model = _LabelRecorder(dp={'rank': rank, 'world': world} if world > 1 else None)
    monkeypatch.setattr(BaseRunner, '_world', staticmethod(lambda m: world))
    torch.manual_seed(7)
    runner.fit(model, data=None, data_processor=_RatingDP(_batches(n_full, ragged)))
    return model


@pytest.mark.parametrize('n_full,ragged', [(5, 3), (4, 0), (3, 1), (0, 5)])
def test_single_process_rating_epoch_carries_its_labels(n_full, ragged, monkeypatch):
    """One process: the full batches run from the resident epoch with their own labels, the ragged tail step by step;
    every batch once, in order, and the draws are the single torch.randint stream of DCCF.py:72."""
    m = _run(n_full, ragged, 1, 0, monkeypatch)
    resident = n_full if n_full + (1 if ragged else 0) > 2 else 0      # (only an epoch of more than two batches)
    assert [int(x[0, 0]) for x, _ in m.resident] == list(range(resident))
    for k, y in enumerate(m.labels):
        assert torch.equal(y, _label(k, 8))
    tail = list(range(resident, n_full)) + ([n_full] if ragged else [])
    assert [int(x[0, 0]) for x, _ in m.stepwise] == tail
    for k, y in zip(tail, m.stepwise_labels):
        assert torch.equal(y, _label(k, y.shape[0]))
    sizes = [8] * n_full + ([ragged] if ragged else [])
    torch.manual_seed(7)
    stream = torch.randint(1000, (sum(sizes), 10))
    assert torch.equal(torch.cat([si for _, si in m.resident + m.stepwise]), stream)


@pytest.mark.parametrize('n_full,ragged,world', [(9, 3, 2), (8, 0, 4), (3, 2, 4), (13, 0, 8), (17, 5, 8)])
def test_data_parallel_rating_epoch_keeps_each_ranks_labels(n_full, ragged, world, monkeypatch):
    """As rank r of `world`: global step k takes batch k*world + r with its own labels (labels are not exchanged: only
    the owning rank's middle kernel reads them); the ranks' draws re-assemble the single stream; what does not fill a
    global step runs step by step with data parallelism suspended, with its labels, identically on every rank."""
    runs = [_run(n_full, ragged, world, r, monkeypatch) for r in range(world)]
    n_steps = n_full // world
    torch.manual_seed(7)
    stream = torch.randint(1000, (n_steps * world * 8, 10)).view(n_steps * world, 8, 10)
    tail = list(range(n_steps * world, n_full)) + ([n_full] if ragged else [])
    for r, m in enumerate(runs):
        assert [int(x[0, 0]) for x, _ in m.resident] == [k * world + r for k in range(n_steps)]
        assert len(m.labels) == n_steps
        for k, ((_, si), y) in enumerate(zip(m.resident, m.labels)):
            assert torch.equal(si, stream[k * world + r])
            assert torch.equal(y, _label(k * world + r, 8))
        assert [int(x[0, 0]) for x, _ in m.stepwise] == tail
        for k, y in zip(tail, m.stepwise_labels):
            assert torch.equal(y, _label(k, y.shape[0]))
        assert all(m.suspended_flags) and m._dp is not None
    for a, b in zip(runs[0].stepwise, runs[-1].stepwise):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.fixture(scope='module')
def lib():
    build.build()
    return _lib.load()


def _fwd_bwd(lib, n_pairs, mse_pairs):
    return lib.dccf_train_fwd_bwd_tc(None, None, None, None, None, None, None, None, None, None, n_pairs, mse_pairs,
                                     None, 1, None, None, None, 0, None, None, None, None, None, None, None, None, None,
                                     None, None, None, None, None, 7, None, None)


def test_mse_pair_count_below_the_batch_is_refused_without_a_gpu(lib):
    """dccf_train_fwd_bwd_tc rejects an MSE pair count below n_pairs before any CUDA call; 0 (this call's pairs) and
    any count >= n_pairs pass that check (and then fail on the missing buffers)."""
    for bad in (1, 63, -1):
        assert _fwd_bwd(lib, 64, bad) == -1
        assert b'mse_pairs' in lib.dccf_last_error(), bad
    for ok in (0, 64, 128):
        assert _fwd_bwd(lib, 64, ok) == -1
        assert b'mse_pairs' not in lib.dccf_last_error(), ok


def test_staged_labels_need_a_staging_launch(lib):
    """dccf_adam_link_ids copies labels only where it stages a batch: Y_out without the epoch arrays is refused."""
    dims = _lib.Dims(n_users=4, n_items=4, dim=64, feat_dim=64, n_samples=1, n_attr=1)
    ids = (ctypes.c_int64 * 16)()
    heads = (ctypes.c_int32 * 16)()
    labels = (ctypes.c_float * 4)()
    extra = _lib.LinkExtra()
    extra.Y_out = ctypes.addressof(labels)
    rc = lib.dccf_adam_link_ids(ctypes.byref(dims), ids, ids, 4, 1, 0, -1, heads, heads, heads, heads, None, None, None,
                                None, None, ctypes.byref(extra), None)
    assert rc == -1 and b'Y_out needs staging' in lib.dccf_last_error()
