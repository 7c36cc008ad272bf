"""Host side of the path (no GPU): DataLoader / DataProcessor / model init / runner bookkeeping compared with
fixtures produced by the unmodified reference (tests/golden/sampler.npz, train_*.npz)."""
import argparse
import os

import numpy as np
import pytest
import torch

from dccf_b200 import synth
from dccf_b200.data_loaders.DataLoader import DataLoader
from dccf_b200.data_processor.DataProcessor import DataProcessor
from dccf_b200.models.DCCF import DCCF
from dccf_b200.runners.BaseRunner import BaseRunner
from dccf_b200.utils import utils

SENT = synth.DEFAULT_SENTENCE_MODEL


def _write_sampler_dataset(g, root):
    d = os.path.join(root, 's')
    os.makedirs(d)
    for split in ('train', 'validation', 'test'):
        np.savetxt(os.path.join(d, 's.%s.csv' % split), g[split + '_csv'], fmt='%d', delimiter=',')
    I, U = int(g['item_num']), int(g['user_num'])
    np.save(os.path.join(d, 's_%s.npy' % SENT), np.zeros((I, 64), np.float32))
    np.save(os.path.join(d, 's.ips_expo_prob.npy'), np.zeros((U, I), np.float32))
    return d


def _make_model(d, dataset, U, I, seed=2019, **kw):
    model = DCCF(path=d, dataset=dataset, sentence_model=SENT, sample_num=kw.get('S', 10),
                 attribute_num=kw.get('A', 2), std=kw.get('std', 0.1), label_min=0, label_max=1, feature_num=0,
                 user_num=U, item_num=I, u_vector_size=64, i_vector_size=64, n_layers=1, random_seed=seed,
                 model_path=os.path.join(d, 'm.pt'))
    model.apply(model.init_paras)
    return model


def test_loader_and_sampler_bit_exact(golden, tmp_path):
    """Same seed -> the same test/validation negatives, epoch shuffles and training negatives, bit for bit
    (src/data_processor/DataProcessor.py:57-111, 227-250, 408-524; src/utils/utils.py:82-92)."""
    g = golden('sampler')
    d = _write_sampler_dataset(g, str(tmp_path))
    seed = int(g['seed'])
    torch.manual_seed(seed)
    np.random.seed(seed)
    dl = DataLoader(path=str(tmp_path), dataset='s', label='label', sep=',')
    assert dl.user_num == int(g['user_num']) and dl.item_num == int(g['item_num'])
    model = _make_model(d, 's', dl.user_num, dl.item_num, seed=seed)
    dl.drop_neg()
    dp = DataProcessor(dl, model, rank=1, test_neg_n=int(g['test_neg_n']))
    te = dp.get_test_data()
    va = dp.get_validation_data()
    for nm, dd in (('test', te), ('validation', va)):
        for k in ('uid', 'iid', 'Y', 'X', 'sample_id'):
            assert np.array_equal(np.asarray(dd[k]), g['%s_%s' % (nm, k)]), (nm, k)
    tr = dp.get_train_data(epoch=-1)
    assert np.array_equal(tr['X'], g['train0_X'])
    for ep in range(int(g['epochs'])):
        data = dp.get_train_data(epoch=ep)
        assert np.array_equal(data['sample_id'], g['train_ep%d_order' % ep])
        batches = dp.prepare_batches(data, int(g['batch_size']), train=True)
        assert len(batches) == int(g['train_ep%d_nbatches' % ep])
        X = np.concatenate([b['X'].cpu().numpy() for b in batches])
        Y = np.concatenate([b['Y'].cpu().numpy() for b in batches])
        sid = np.concatenate([b['sample_id'] for b in batches])
        assert np.array_equal(X, g['train_ep%d_X' % ep])                 # negatives bit-exact
        assert np.array_equal(Y, g['train_ep%d_Y' % ep])
        assert np.array_equal(sid, g['train_ep%d_sample_id' % ep])
        for b in batches:                                                 # layout contract (DP:160-207)
            r = b['real_batch_size']
            assert b['X'].shape[0] == 2 * r and b['total_batch_size'] == 2 * r
            assert torch.equal(b['X'][:r, 0], b['X'][r:, 0])
    assert np.array_equal(np.random.get_state()[1][:8].astype(np.int64), g['np_state_after'])


def test_eval_batches_are_cached_and_plain(golden, tmp_path):
    g = golden('sampler')
    d = _write_sampler_dataset(g, str(tmp_path))
    np.random.seed(1)
    dl = DataLoader(path=str(tmp_path), dataset='s', label='label', sep=',')
    model = _make_model(d, 's', dl.user_num, dl.item_num)
    dl.drop_neg()
    dp = DataProcessor(dl, model, rank=1, test_neg_n=3)
    te = dp.get_test_data()
    b1 = dp.prepare_batches(te, 50, train=False)
    b2 = dp.prepare_batches(te, 50, train=False)
    assert b1 is b2
    assert all(b['rank'] == 1 for b in b1)
    assert sum(b['X'].shape[0] for b in b1) == len(te['Y'])
    # one negative set per distinct user (DP:420-430)
    n_users = len(set(te['uid'].tolist()))
    assert int((te['Y'] == 0).sum()) == 3 * n_users


@pytest.mark.parametrize('name', ['train_f64', 'train_f768'])
def test_initial_weights_equal_reference(golden, tmp_path, name):
    """Same constructor order + apply(init_paras) on the torch CPU generator -> identical initial parameters
    (src/models/DCCF.py:47-64, src/models/BaseModel.py:131-151, src/main.py:150)."""
    g = golden(name)
    U, I = g['init_E_user'].shape[0], g['init_E_item'].shape[0]
    d = str(tmp_path)
    np.save(os.path.join(d, 'g_%s.npy' % SENT), g['feat'])
    np.save(os.path.join(d, 'g.ips_expo_prob.npy'), g['expo'])
    seed = int(g['seed'])
    torch.manual_seed(seed)
    model = _make_model(d, 'g', U, I, seed=seed)
    assert np.array_equal(model.uid_embeddings.weight.detach().numpy(), g['init_E_user'])
    assert np.array_equal(model.iid_embeddings.weight.detach().numpy(), g['init_E_item'])
    assert np.array_equal(model.mlp[0].weight.detach().numpy(), g['init_W'])
    assert np.array_equal(model.mlp[0].bias.detach().numpy(), g['init_b'])
    assert sorted(model.state_dict().keys()) == ['iid_embeddings.weight', 'mlp.0.bias', 'mlp.0.weight',
                                                 'uid_embeddings.weight']
    assert model.total_parameters == (U + I) * 64 + 64 * (64 + g['feat'].shape[1]) + 64


def test_model_refuses_cpu(golden, tmp_path):
    """No CPU fallback: predict on a CPU model must fail loudly, whether or not the machine has a GPU."""
    g = golden('train_f64')
    d = str(tmp_path)
    np.save(os.path.join(d, 'g_%s.npy' % SENT), g['feat'])
    np.save(os.path.join(d, 'g.ips_expo_prob.npy'), g['expo'])
    model = _make_model(d, 'g', 40, 50)
    with pytest.raises(RuntimeError, match='CUDA only'):
        model.predict({'X': torch.from_numpy(g['X_0']), 'dropout': 0.0})


def test_cli_flags_and_defaults():
    """Appendix A of SURVEY.md: flag names and defaults of the reference CLI."""
    p = argparse.ArgumentParser()
    utils.parse_global_args(p)
    DataLoader.parse_data_args(p)
    DCCF.parse_model_args(p, model_name='DCCF')
    BaseRunner.parse_runner_args(p)
    DataProcessor.parse_dp_args(p)
    a = p.parse_args([])
    assert (a.gpu, a.random_seed, a.train) == ('0', 2019, 1)
    assert (a.path, a.dataset, a.sep, a.label) == ('../datasets/', 'ml100k-1-5', ',', 'label')
    assert (a.u_vector_size, a.i_vector_size, a.n_layers) == (64, 64, 1)
    assert (a.sentence_model, a.sample_num, a.attribute_num, a.std) == ('paraphrase-distilroberta-base-v1', 10, 2, 0.1)
    assert (a.optimizer, a.lr, a.l2, a.batch_size, a.eval_batch_size, a.dropout) == ('GD', 0.01, 1e-4, 128, 16384, 0.2)
    assert (a.epoch, a.check_epoch, a.early_stop, a.skip_eval, a.load, a.metric) == (100, 1, 1, 0, 0, 'RMSE')
    assert a.test_neg_n == 100
    assert a.model_path == '../model/DCCF/DCCF.pt'
    assert (DCCF.append_id, DCCF.include_id, DCCF.include_user_features, DCCF.include_item_features,
            DCCF.include_context_features) == (True, False, False, False, False)


def test_utils_behaviour():
    assert utils.format_metric([0.123456, np.float32(0.5), 3]) == '0.1235,0.5000,3'
    assert utils.best_result('ndcg@5', [[0.1, 0.9], [0.2, 0.0]]) == [0.2, 0.0]       # lexicographic (utils.py:95-106)
    assert utils.best_result('rmse', [3.0, 1.0, 2.0]) == 1.0
    np.random.seed(3)
    data = {'a': np.arange(10), 'b': np.arange(10) * 2, 'c': np.stack([np.arange(10), np.arange(10)], 1)}
    utils.shuffle_in_unison_scary(data)
    assert np.array_equal(data['b'], data['a'] * 2) and np.array_equal(data['c'][:, 0], data['a'])
    assert not np.array_equal(data['a'], np.arange(10))


def test_runner_bookkeeping():
    r = BaseRunner(optimizer='Adam', learning_rate=1e-3, metrics='NDCG@5,Recall@5', dropout=0.2)
    assert r.metrics == ['ndcg@5', 'recall@5']
    batches = r.batches_add_control([{}, {}], train=True)
    assert all(b['dropout'] == 0.2 and b['train'] for b in batches)
    batches = r.batches_add_control([{}], train=False)
    assert batches[0]['dropout'] == 0.0 and not batches[0]['train']
    r.valid_results = [[0.5]] + [[0.1]] * 21
    assert r.eva_termination(None)            # best result more than 20 evaluations ago


def test_native_sampler_equals_python_loop(golden, tmp_path):
    """dccf_sample_negatives (C++) consumes numpy's MT19937 stream exactly like the Python loop that mirrors
    src/data_processor/DataProcessor.py:446-524: same negatives, same generator state afterwards — on the
    golden dataset (both sampler branches) and on a random one."""
    g = golden('sampler')
    d = _write_sampler_dataset(g, str(tmp_path))
    dl = DataLoader(path=str(tmp_path), dataset='s', label='label', sep=',')
    model = _make_model(d, 's', dl.user_num, dl.item_num)
    dl.drop_neg()
    results = []
    for native in (False, True):
        np.random.seed(77)
        dp = DataProcessor(dl, model, rank=1, test_neg_n=int(g['test_neg_n']))
        dp.use_native_sampler = native
        te = dp.get_test_data()
        xs = [te['X'].copy()]
        for ep in range(3):
            data = dp.get_train_data(epoch=ep)
            batches = dp.prepare_batches(data, 16, train=True)
            xs.append(np.concatenate([b['X'].cpu().numpy() for b in batches]))
        results.append((xs, np.random.get_state()[1].copy(), np.random.get_state()[2]))
    for a, b in zip(results[0][0], results[1][0]):
        assert np.array_equal(a, b)
    assert np.array_equal(results[0][1], results[1][1]) and results[0][2] == results[1][2]


def test_native_sampler_reports_exhausted_user(tmp_path):
    """The reference asserts `remain_iids_num >= neg_n` (DataProcessor.py:495); so does the native sampler."""
    from dccf_b200 import synth
    d = synth.write_dataset(str(tmp_path), 'x', n_users=5, n_items=40, per_user=10, feat_dim=64, seed=3)
    dl = DataLoader(path=str(tmp_path), dataset='x', label='label', sep=',')
    model = _make_model(d, 'x', dl.user_num, dl.item_num)
    dl.drop_neg()
    dp = DataProcessor(dl, model, rank=1, test_neg_n=35)
    with pytest.raises(AssertionError):
        dp.get_test_data()


def test_array_route_equals_dataframe_route(golden, tmp_path):
    """The id-only shortcut of DataProcessor (data dicts and epochs assembled from arrays) yields exactly what the
    reference-shaped DataFrame route (generate_neg_df -> concat -> format_data_dict, DP:73-111,227-250,292-356,
    408-444) yields: every key, dtype and value of the test / validation dicts, every batch of three epochs
    including a ragged last batch, and the numpy generator afterwards."""
    g = golden('sampler')
    d = _write_sampler_dataset(g, str(tmp_path))
    dl = DataLoader(path=str(tmp_path), dataset='s', label='label', sep=',')
    model = _make_model(d, 's', dl.user_num, dl.item_num)
    dl.drop_neg()
    runs = []
    for fast in (False, True):
        np.random.seed(5)
        dp = DataProcessor(dl, model, rank=1, test_neg_n=int(g['test_neg_n']))
        dp.fast_ids_path = fast
        te, va = dp.get_test_data(), dp.get_validation_data()
        epochs = []
        for ep in range(3):
            data = dp.get_train_data(epoch=ep)
            assert len(data['Y']) % 13 != 0                              # the last batch is ragged
            epochs.append(dp.prepare_batches(data, 13, train=True))
        runs.append((te, va, epochs, np.random.get_state()))
    slow, fast = runs
    for a, b in ((slow[0], fast[0]), (slow[1], fast[1])):
        assert sorted(a.keys()) == sorted(b.keys())
        for k in a:
            assert np.asarray(a[k]).dtype == np.asarray(b[k]).dtype and np.array_equal(a[k], b[k]), k
    for ea, eb in zip(slow[2], fast[2]):
        assert len(ea) == len(eb)
        for ba, bb in zip(ea, eb):
            assert sorted(ba.keys()) == sorted(bb.keys())
            for k in ba:
                if torch.is_tensor(ba[k]):
                    assert ba[k].dtype == bb[k].dtype and torch.equal(ba[k], bb[k]), k
                else:
                    assert np.array_equal(ba[k], bb[k]), k
    assert np.array_equal(slow[3][1], fast[3][1]) and slow[3][2] == fast[3][2]


@pytest.mark.parametrize('n', [1, 2, 257, 5000])
def test_one_pass_shuffle_equals_replayed_shuffle(n):
    """shuffle_in_unison_scary applies ONE permutation; the reference replays the generator state per array
    (src/utils/utils.py:82-92).  Same arrays, same identity (in place), same generator state afterwards."""
    rs = np.random.RandomState(n)
    base = {'uid': rs.randint(0, 50, n), 'Y': rs.rand(n).astype(np.float32),
            'X': rs.randint(0, 99, (n, 2)), 'sample_id': np.arange(n)}
    ref = {k: v.copy() for k, v in base.items()}
    np.random.seed(11)
    state = np.random.get_state()
    for k in ref:                                   # the reference's loop, literally
        np.random.set_state(state)
        np.random.shuffle(ref[k])
    ref_state = np.random.get_state()
    ours = {k: v.copy() for k, v in base.items()}
    ids = {k: id(v) for k, v in ours.items()}
    np.random.seed(11)
    utils.shuffle_in_unison_scary(ours)
    for k in ref:
        assert np.array_equal(ref[k], ours[k]) and id(ours[k]) == ids[k], k
    st = np.random.get_state()
    assert np.array_equal(st[1], ref_state[1]) and st[2] == ref_state[2]
    # arrays that alias each other or differ in length take the literal replay
    np.random.seed(11)
    x = np.arange(10)
    odd = {'a': x, 'b': x[::-1], 'c': np.arange(4)}
    utils.shuffle_in_unison_scary(odd)


def test_history_grouping_equals_groupby_loop():
    """group_user_interactions_df (src/utils/mining.py:18-29): same frame as the reference's per-group loop —
    ascending uid, items in file order, non-positive labels dropped, users without positives absent."""
    import pandas as pd
    from dccf_b200.utils.mining import group_user_interactions_df
    rs = np.random.RandomState(4)
    df = pd.DataFrame({'uid': rs.randint(0, 40, 500), 'iid': rs.randint(0, 90, 500), 'label': rs.randint(0, 2, 500),
                       'time': np.arange(500)})
    uids, inters = [], []
    for uid, group in df[df['label'] > 0].groupby('uid'):          # the reference's loop
        uids.append(uid)
        inters.append(','.join(str(i) for i in group['iid'].tolist()))
    got = group_user_interactions_df(df, label='label', seq_sep=',')
    assert got['uid'].tolist() == uids and got['iids'].tolist() == inters
    assert list(got.columns) == ['uid', 'iids']
    empty = group_user_interactions_df(df[df['label'] > 5], label='label')
    assert len(empty) == 0 and list(empty.columns) == ['uid', 'iids']


def test_data_order_is_recognised_from_addresses():
    want = np.arange(100)
    slices = [{'sample_id': want[a:a + 30]} for a in range(0, 100, 30)]
    assert BaseRunner._slices_of(slices, want)
    assert not BaseRunner._slices_of(slices[:-1], want)                       # incomplete
    assert not BaseRunner._slices_of(slices[::-1], want)                      # out of order
    assert not BaseRunner._slices_of([{'sample_id': want.copy()}], want)      # equal values, other memory
    assert not BaseRunner._slices_of([{'sample_id': want[::2]}, {'sample_id': want[1::2]}], want)


@pytest.mark.parametrize('item_num', [1, 2, 16000, 999983, (1 << 28) - 1])
def test_confounder_draw_equals_torch_randint(item_num):
    """dccf_confounder_draw replays `torch.randint(item_num, size=(P, S))` (src/models/DCCF.py:72) on the torch CPU
    generator: the same ids AND the same generator afterwards (other consumers continue unchanged) — from a freshly
    seeded generator, from mid-generation positions, across generation boundaries, interleaved with torch's own draws."""
    from dccf_b200 import host_rng
    assert host_rng.available()
    torch.manual_seed(2019)
    want = [torch.randint(item_num, (256, 10)), torch.randint(item_num, (16384, 10)), torch.rand(7),
            torch.randint(item_num, (37, 10)), torch.randint(item_num, (1, 1)), torch.randn(5),
            torch.randint(item_num, (624 * 3,))]
    state_want = torch.get_rng_state()
    torch.manual_seed(2019)
    got = [host_rng.randint(item_num, (256, 10), min_draws=0), host_rng.randint(item_num, (16384, 10)), torch.rand(7),
           host_rng.randint(item_num, (37, 10), min_draws=0), host_rng.randint(item_num, (1, 1), min_draws=0),
           torch.randn(5), host_rng.randint(item_num, (624 * 3,), min_draws=0)]
    for a, b in zip(want, got):
        assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)
    assert torch.equal(state_want, torch.get_rng_state())


def test_confounder_draw_leaves_other_cases_to_torch():
    """Ranges where torch draws 64-bit words (>= 2^28), small draws and private generators still give torch's numbers."""
    from dccf_b200 import host_rng
    g1, g2 = torch.Generator(), torch.Generator()
    g1.manual_seed(9)
    g2.manual_seed(9)
    for high, n in ((1 << 28, 20000), ((1 << 31) + 5, 20000), (16000, 50000), (16000, 3)):
        assert torch.equal(torch.randint(high, (n,), generator=g1), host_rng.randint(high, (n,), generator=g2))
    assert torch.equal(g1.get_state(), g2.get_state())


def test_model_draws_confounders_like_the_reference(golden, tmp_path):
    """DCCF.draw_confounders == the torch.randint call of DCCF.py:72, for a training batch and an evaluation batch."""
    g = golden('train_f64')
    d = str(tmp_path)
    np.save(os.path.join(d, 'g_%s.npy' % SENT), g['feat'])
    np.save(os.path.join(d, 'g.ips_expo_prob.npy'), g['expo'])
    model = _make_model(d, 'g', 40, 50)
    torch.manual_seed(4)
    want = [torch.randint(50, (256, 10)), torch.randint(50, (16384, 10))]
    torch.manual_seed(4)
    got = [model.draw_confounders(256), model.draw_confounders(16384)]
    assert all(torch.equal(a, b) for a, b in zip(want, got))


@pytest.mark.parametrize('F,degenerate', [(768, False), (64, False), (128, True)])
def test_projection_factor_reproduces_the_noise_covariance(golden, tmp_path, F, degenerate):
    """DCCF.projection_factor: M with M·M^T = W_f·W_f^T, so that M·g (g ~ N(0, std^2 I_64)) is distributed like the
    reference's W_f·eps (eps ~ N(0, std^2 I_F), src/models/DCCF.py:87-92) — also when W_f has deficient rank."""
    d = str(tmp_path)
    rs = np.random.RandomState(F)
    np.save(os.path.join(d, 'g_%s.npy' % SENT), rs.standard_normal((50, F)).astype(np.float32))
    np.save(os.path.join(d, 'g.ips_expo_prob.npy'), rs.random_sample((40, 50)).astype(np.float32))
    model = _make_model(d, 'g', 40, 50)
    with torch.no_grad():
        model.mlp[0].weight.copy_(torch.from_numpy(rs.standard_normal((64, 64 + F)).astype(np.float32)))
        if degenerate:
            model.mlp[0].weight[5] = model.mlp[0].weight[3]           # two equal rows: rank 63
            model.mlp[0].weight[9, 64:] = 0.0                         # a row of W_f that is zero
    Wf = model.mlp[0].weight.detach()[:, 64:].double().numpy()
    M = model.projection_factor().numpy()
    cov = Wf @ Wf.T
    assert M.shape == (64, 64) and np.isfinite(M).all()
    assert np.abs(M @ M.T - cov).max() < 1e-10 * np.abs(cov).max()
    # sampled check of the law itself: cov(M g) == cov(W_f eps) == std^2 W_f W_f^T
    g = rs.standard_normal((200000, 64)) * 0.1
    emp = (g @ M.T).T @ (g @ M.T) / len(g)
    assert np.abs(emp - 0.01 * cov).max() < 0.02 * 0.01 * np.abs(cov).max()


def test_device_confounder_schedule_emulated(tmp_path):
    """k_confounder_draw (MT19937 continued on the device, three barrier-separated phases per generation) cannot run
    here, but its per-phase functions are plain C++ (dccf_b200/csrc/mt19937.cuh): tests/mt_emulate.cpp executes them
    for every thread of the CTA in forward, backward and shuffled order and compares ids, final words and position with
    the textbook sequential generator over 400 random states / positions / counts / ranges."""
    import shutil
    import subprocess
    from conftest import ROOT
    gxx = shutil.which('g++')
    if gxx is None:
        pytest.skip('g++ not available')
    exe = str(tmp_path / 'mt_emulate')
    subprocess.run([gxx, '-O2', '-std=c++17', '-o', exe, os.path.join(ROOT, 'tests', 'mt_emulate.cpp')], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and 'MT_EMULATION_OK' in r.stdout, r.stdout + r.stderr


def test_device_stream_state_round_trip_without_draws():
    """host_rng.DeviceStream packs torch's generator as [624 words | next unread index] and restores it: with no draw in
    between the generator is exactly where it was (checked on a CPU 'device'; the kernel itself needs a GPU)."""
    from dccf_b200 import host_rng
    for prep in (lambda g: None, lambda g: torch.randint(50, (1000,), generator=g), lambda g: torch.randn(3, generator=g)):
        g1, g2 = torch.Generator(), torch.Generator()
        g1.manual_seed(5)
        g2.manual_seed(5)
        prep(g1)
        prep(g2)
        s = host_rng.DeviceStream('cpu', generator=g2)
        packed = s.state.numpy().view(np.uint32)
        assert packed.shape == (625,) and 0 <= int(packed[624]) <= 624
        s.finish()
        assert torch.equal(torch.randint(1 << 20, (700,), generator=g1), torch.randint(1 << 20, (700,), generator=g2))
        assert torch.equal(torch.randn(5, generator=g1), torch.randn(5, generator=g2))


def test_config0_host_pipeline_digest(tmp_path):
    """BASELINE.json configs[0] — 2 000 users x 5 000 items x 768-d, test_neg_n = 1000, batch 128 — the host side of the
    path against the UNMODIFIED reference at full size: the reference's own DataLoader / DataProcessor produced
    tests/golden/config0_digest.json (oracle/make_golden.py::make_config0_digest; 2 M negatives per evaluation set, so
    sha256 digests instead of the arrays).  Every id, label and sample id of the test / validation sets and of two
    shuffled training epochs, and the numpy generator afterwards, must match bit for bit."""
    import hashlib
    import json
    from conftest import GOLDEN
    want = json.load(open(os.path.join(GOLDEN, 'config0_digest.json')))

    def digest(a):
        a = np.ascontiguousarray(a)
        h = hashlib.sha256()
        h.update(str(a.dtype).encode() + b'|' + str(a.shape).encode() + b'|')
        h.update(a.tobytes())
        return h.hexdigest()

    d = synth.write_dataset(str(tmp_path), 'tiny', want['users'], want['items'], want['per_user'],
                            feat_dim=64, seed=want['seed'])       # the feature width does not enter the host pipeline
    seed = want['seed']
    torch.manual_seed(seed)
    np.random.seed(seed)
    dl = DataLoader(path=str(tmp_path), dataset='tiny', label='label', sep=',')
    assert (int(dl.user_num), int(dl.item_num)) == (want['user_num'], want['item_num'])
    for fname, sha in want['files'].items():         # .info.json and the two history files: byte for byte
        assert hashlib.sha256(open(os.path.join(d, fname), 'rb').read()).hexdigest() == sha, fname
    model = _make_model(d, 'tiny', dl.user_num, dl.item_num, seed=seed)
    dl.drop_neg()
    dp = DataProcessor(dl, model, rank=1, test_neg_n=want['test_neg_n'])
    te, va = dp.get_test_data(), dp.get_validation_data()
    for nm, dd in (('test', te), ('validation', va)):
        assert len(dd['Y']) == want['rows'][nm]
        for k in ('uid', 'iid', 'Y', 'X', 'sample_id'):
            assert digest(np.asarray(dd[k])) == want['digests']['%s_%s' % (nm, k)], (nm, k)
    dp.get_train_data(epoch=-1)
    for ep in range(want['epochs']):
        data = dp.get_train_data(epoch=ep)
        batches = dp.prepare_batches(data, want['batch_size'], train=True)
        assert len(batches) == want['rows']['train_ep%d_batches' % ep]
        assert digest(np.concatenate([b['X'].cpu().numpy() for b in batches])) == want['digests']['train_ep%d_X' % ep]
        assert digest(np.concatenate([b['Y'].cpu().numpy() for b in batches])) == want['digests']['train_ep%d_Y' % ep]
        sid = np.concatenate([np.asarray(b['sample_id']) for b in batches]).astype(np.int64)
        assert digest(sid) == want['digests']['train_ep%d_sample_id' % ep]
    assert [int(x) for x in np.random.get_state()[1][:8]] == want['np_state_after']


@pytest.mark.parametrize('fixture', ['run_recmodel', 'run_recmodel_rank0'])
def test_whole_run_equals_reference_run(golden, tmp_path, fixture, monkeypatch):
    """src/main.py's whole sequence with the mirrored classes == the same sequence of the UNMODIFIED reference
    (tests/golden/run_recmodel.npz, oracle/make_golden.py::make_run_fixture; RecModel on CPU so that every number is
    reproducible): "Test Before Training", the per-epoch train / validation / test metric lists of runner.train (i.e.
    shuffles, negatives, Adam steps with l2 + clip, evaluation, model selection and the reload of the best epoch),
    "Test After Training", the final predictions and the checkpointed parameters."""
    from dccf_b200.models.RecModel import RecModel
    # the reference ran with no CUDA device visible (oracle/ref_harness.py::cpu_shims): so does the mirrored pipeline,
    # which would otherwise move the batches of this CPU model to a GPU of the machine
    monkeypatch.setattr(torch.cuda, 'device_count', lambda: 0)
    g = golden(fixture)           # rank 1: top-n recommendation (BPR, sampled negatives); rank 0: rating prediction (MSE)
    seed, rank = int(g['seed']), int(g['rank'])
    synth.write_dataset(str(tmp_path), 'toy', int(g['n_users']), int(g['n_items']), int(g['per_user']), feat_dim=64,
                        seed=seed + 5)
    model_path = str(tmp_path / 'model' / 'm.pt')
    import logging
    import re
    messages = []

    class Collect(logging.Handler):
        def emit(self, record):
            messages.append(record.getMessage())

    collector = Collect(level=logging.INFO)
    root_logger = logging.getLogger()
    old_level = root_logger.level
    root_logger.addHandler(collector)
    root_logger.setLevel(logging.INFO)
    torch.manual_seed(seed)
    np.random.seed(seed)
    dl = DataLoader(path=str(tmp_path), dataset='toy', label='label', sep=',')
    model = RecModel(label_min=dl.label_min, label_max=dl.label_max, feature_num=0, user_num=dl.user_num,
                     item_num=dl.item_num, u_vector_size=64, i_vector_size=64, random_seed=seed, model_path=model_path)
    model.apply(model.init_paras)
    if rank == 1:
        dl.drop_neg()
    dp = DataProcessor(dl, model, rank=rank, test_neg_n=int(g['test_neg_n']))
    runner = BaseRunner(optimizer='Adam', learning_rate=float(g['lr']), epoch=int(g['epochs']),
                        batch_size=int(g['batch_size']), eval_batch_size=16384, dropout=0.2, l2=float(g['l2']),
                        metrics='rmse,mae', check_epoch=1, early_stop=1)
    runner.show_progress = False
    before = runner.evaluate(model, dp.get_test_data(), dp)
    runner.train(model, dp, skip_eval=0)
    after = runner.evaluate(model, dp.get_test_data(), dp, write_rank=True)
    pred = runner.predict(model, dp.get_test_data(), dp)
    root_logger.removeHandler(collector)
    root_logger.setLevel(old_level)
    # the log: same lines in the same order, same wording, same %.4f numbers (durations masked)
    keep = ('load ', 'size of ', 'label:', '# of ', 'Model # of', 'Drop Neg', 'Prepare ', 'Optimizer:', 'Init:', 'Epoch ',
            'Best Iter', 'Early stop', 'Save model', 'Load model', 'building ', 'loss = ', 'l2 inappropriate', 'Test Before', 'Test After', 'Save Test Results', '# cuda devices',
            'DataLoader:', 'Model:', 'Runner:', 'DataProcessor:')
    ours = [re.sub(r'\[\d+\.\d+ s\]', '[T s]', m.strip().replace(str(tmp_path), '<root>')) for m in messages
            if m.strip().startswith(keep)]
    assert ours == [str(x) for x in g['log']]
    # rank.csv (BaseRunner.py:315-323): tab separated uid / iid / score / label, sorted by uid
    lines = open(os.path.join(dl.path, 'rank.csv')).read().strip().split(chr(10))
    assert lines[0] == str(g['rank_header'])
    rows = np.array([[float(x) for x in ln.split(chr(9))] for ln in lines[1:]])
    assert rows.shape == g['rank_rows'].shape
    assert np.array_equal(rows[:, [0, 1, 3]], g['rank_rows'][:, [0, 1, 3]])
    assert np.abs(rows[:, 2] - g['rank_rows'][:, 2]).max() <= 1e-6 * np.abs(g['rank_rows'][:, 2]).max()
    assert np.allclose(before, g['before'], rtol=1e-6, atol=0)
    for ours, name in ((runner.train_results, 'train_results'), (runner.valid_results, 'valid_results'),
                       (runner.test_results, 'test_results')):
        assert np.asarray(ours).shape == g[name].shape and np.allclose(ours, g[name], rtol=1e-6, atol=0), name
    assert np.allclose(after, g['after'], rtol=1e-6, atol=0)
    assert np.abs(pred - g['pred']).max() <= 1e-6 * np.abs(g['pred']).max()
    sd = model.state_dict()
    assert sorted('sd_' + k for k in sd) == sorted(k for k in g.files if k.startswith('sd_'))
    for k, v in sd.items():
        assert np.abs(v.numpy() - g['sd_' + k]).max() <= 1e-6 * np.abs(g['sd_' + k]).max(), k


def test_whole_dccf_run_orchestration_on_cpu(golden, tmp_path, monkeypatch):
    """tests/golden/run_dccf.npz (a whole DCCF run of the unmodified reference, --std 0 --dropout 0) replayed on CPU
    with the MIRRORED loader, processor and runner around a stand-in for the device math (oracle/torch_port.py, the
    eager-torch port): every shuffle, negative, confounder draw, evaluation pass, Adam step, model selection and reload
    happens in the reference's order — "before", per-epoch and "after" metrics, predictions and checkpoint agree to 1e-5.
    (The GPU path replays the same fixture in tests/test_gpu_parity.py::test_whole_dccf_run_equals_reference_run.)"""
    from oracle import dccf_oracle as O
    from oracle import torch_port
    monkeypatch.setattr(torch.cuda, 'device_count', lambda: 0)     # CPU replay on any machine, see above

    class PortModel(torch_port.DCCFPort):
        append_id, include_id = True, False
        include_user_features = include_item_features = include_context_features = False
        optimizer = None

        def predict(self, feed_dict):
            fd = dict(feed_dict)
            fd['noise'] = 0.0               # --std 0: the reference's zero noise comes off the CUDA generator, not this one
            return torch_port.DCCFPort.predict(self, fd)

        def save_model(self, model_path=None):
            os.makedirs(os.path.dirname(self.model_path), exist_ok=True)
            torch.save(self.state_dict(), self.model_path)

        def load_model(self, model_path=None):
            self.load_state_dict(torch.load(self.model_path))
            self.eval()

        @staticmethod
        def evaluate_method(p, data, metrics):
            p = p.detach().numpy() if torch.is_tensor(p) else np.asarray(p)
            out = []
            for m in metrics:
                d = np.asarray(data['Y'], np.float64) - p.astype(np.float64)
                out.append(float(np.sqrt(np.mean(d * d))) if m == 'rmse' else float(np.mean(np.abs(d))) if m == 'mae'
                           else O.evaluate_method(p, data, [m])[0])
            return out

    g = golden('run_dccf')
    seed = int(g['seed'])
    d = synth.write_dataset(str(tmp_path), 'toy', int(g['n_users']), int(g['n_items']), int(g['per_user']), feat_dim=64,
                            seed=seed + 5)
    torch.manual_seed(seed)
    np.random.seed(seed)
    dl = DataLoader(path=str(tmp_path), dataset='toy', label='label', sep=',')
    feat = np.load(os.path.join(d, 'toy_%s.npy' % SENT))
    expo = np.load(os.path.join(d, 'toy.ips_expo_prob.npy'))
    model = PortModel(dl.user_num, dl.item_num, feat, expo, sample_num=10, attribute_num=2, std=0.0, seed=seed)
    model.model_path = str(tmp_path / 'model' / 'm.pt')
    dl.drop_neg()
    dp = DataProcessor(dl, model, rank=1, test_neg_n=int(g['test_neg_n']))
    runner = BaseRunner(optimizer='Adam', learning_rate=float(g['lr']), epoch=int(g['epochs']),
                        batch_size=int(g['batch_size']), eval_batch_size=16384, dropout=0.0, l2=float(g['l2']),
                        metrics='ndcg@5,recall@5,precision@5', check_epoch=1, early_stop=1)
    runner.show_progress = False
    before = runner.evaluate(model, dp.get_test_data(), dp)
    runner.train(model, dp, skip_eval=0)
    after = runner.evaluate(model, dp.get_test_data(), dp)
    pred = runner.predict(model, dp.get_test_data(), dp)
    assert np.abs(np.array(before) - g['before']).max() < 1e-6
    for ours, name in ((runner.train_results, 'train_results'), (runner.valid_results, 'valid_results'),
                       (runner.test_results, 'test_results')):
        assert np.asarray(ours).shape == g[name].shape and np.abs(np.asarray(ours) - g[name]).max() < 1e-6, name
    assert np.abs(np.array(after) - g['after']).max() < 1e-6
    assert np.abs(pred - g['pred']).max() <= 1e-5 * np.abs(g['pred']).max()
    for k, v in model.state_dict().items():
        assert np.abs(v.numpy() - g['sd_' + k]).max() <= 1e-5 * np.abs(g['sd_' + k]).max(), k


def test_whole_dccf_run_fused_orchestration_on_cpu(golden, tmp_path):
    """The same fixture through the branches of BaseRunner / DataProcessor that only the CUDA model takes — the
    device-resident epoch of `fit` (one confounder draw per chunk of batches, ragged tail step by step), `train_step`,
    `predict_many` (DCCF's own method, worker-thread draws through dccf_confounder_draw) — with the device math replaced
    by the eager-torch port and the batches merely claiming to live on the GPU.  Same metrics, predictions and checkpoint
    as the reference run: the orchestration the GPU test relies on is exact."""
    from oracle import dccf_oracle as O
    from oracle import torch_port
    from dccf_b200 import host_rng

    class OnDevice(torch.Tensor):
        is_cuda = property(lambda self: True)

    class FusedState(object):                       # what make_fused_optimizer hands the runner: not a torch Optimizer
        def __init__(self, model, lr, l2, weight_decay):
            self.l2 = l2
            self.adam = torch.optim.Adam(model.parameters(), lr=lr, weight_decay=weight_decay)

    class PortModel(torch_port.DCCFPort):
        append_id, include_id = True, False
        include_user_features = include_item_features = include_context_features = False
        optimizer = None
        device_confounders = False
        predict_many = DCCF.predict_many            # the product method itself

        def predict(self, feed_dict):
            fd = dict(feed_dict)
            fd['noise'] = 0.0
            fd['X'] = torch.Tensor(fd['X']).long() if isinstance(fd['X'], OnDevice) else fd['X']
            return torch_port.DCCFPort.predict(self, fd)

        def make_fused_optimizer(self, lr, l2, weight_decay=None):
            return FusedState(self, lr, l2, l2 if weight_decay is None else weight_decay)

        def draw_confounders(self, n_pairs):
            return host_rng.randint(self.item_num, (n_pairs, self.sample_num), min_draws=0)

        def train_step(self, fd):
            fd = dict(fd)
            fd['Y'] = torch.cat([torch.ones(fd['X'].shape[0] // 2), torch.zeros(fd['X'].shape[0] // 2)])
            return torch_port.fit_step(self, self.optimizer.adam, fd, self.optimizer.l2)

        def begin_resident_epoch(self, X_epoch, sample_epoch, dropout):
            state = {'k': 0}
            n = X_epoch.shape[0]

            def step():
                k = state['k']
                state['k'] += 1
                return self.train_step({'X': X_epoch[k], 'sample_item': sample_epoch[k], 'dropout': dropout})
            step.remaining = lambda: n - state['k']
            step.first = None
            return step

        def save_model(self, model_path=None):
            os.makedirs(os.path.dirname(self.model_path), exist_ok=True)
            torch.save(self.state_dict(), self.model_path)

        def load_model(self, model_path=None):
            self.load_state_dict(torch.load(self.model_path))
            self.eval()

        @staticmethod
        def evaluate_method(p, data, metrics):
            p = p.detach().numpy() if torch.is_tensor(p) else np.asarray(p)
            out = []
            for m in metrics:
                d = np.asarray(data['Y'], np.float64) - p.astype(np.float64)
                out.append(float(np.sqrt(np.mean(d * d))) if m == 'rmse' else float(np.mean(np.abs(d))) if m == 'mae'
                           else O.evaluate_method(p, data, [m])[0])
            return out

    class DeviceDP(DataProcessor):
        def _epoch_views(self, rows_X, rows_Y, bounds):
            X = torch.Tensor._make_subclass(OnDevice, torch.from_numpy(np.ascontiguousarray(rows_X)))
            Y = torch.from_numpy(np.ascontiguousarray(rows_Y))
            return [(X[a:b], Y[a:b]) for a, b in bounds]

    g = golden('run_dccf')
    seed = int(g['seed'])
    d = synth.write_dataset(str(tmp_path), 'toy', int(g['n_users']), int(g['n_items']), int(g['per_user']), feat_dim=64,
                            seed=seed + 5)
    torch.manual_seed(seed)
    np.random.seed(seed)
    dl = DataLoader(path=str(tmp_path), dataset='toy', label='label', sep=',')
    model = PortModel(dl.user_num, dl.item_num, np.load(os.path.join(d, 'toy_%s.npy' % SENT)),
                      np.load(os.path.join(d, 'toy.ips_expo_prob.npy')), sample_num=10, attribute_num=2, std=0.0, seed=seed)
    model.model_path = str(tmp_path / 'model' / 'm.pt')
    dl.drop_neg()
    dp = DeviceDP(dl, model, rank=1, test_neg_n=int(g['test_neg_n']))
    runner = BaseRunner(optimizer='Adam', learning_rate=float(g['lr']), epoch=int(g['epochs']),
                        batch_size=int(g['batch_size']), eval_batch_size=16384, dropout=0.0, l2=float(g['l2']),
                        metrics='ndcg@5,recall@5,precision@5', check_epoch=1, early_stop=1)
    runner.show_progress = False
    before = runner.evaluate(model, dp.get_test_data(), dp)
    runner.train(model, dp, skip_eval=0)
    after = runner.evaluate(model, dp.get_test_data(), dp)
    pred = runner.predict(model, dp.get_test_data(), dp)
    assert not isinstance(model.optimizer, torch.optim.Optimizer)          # the fused branch was taken
    assert np.abs(np.array(before) - g['before']).max() < 1e-6
    for ours, name in ((runner.train_results, 'train_results'), (runner.valid_results, 'valid_results'),
                       (runner.test_results, 'test_results')):
        assert np.asarray(ours).shape == g[name].shape and np.abs(np.asarray(ours) - g[name]).max() < 1e-6, name
    assert np.abs(np.array(after) - g['after']).max() < 1e-6
    assert np.abs(pred - g['pred']).max() <= 1e-5 * np.abs(g['pred']).max()
    for k, v in model.state_dict().items():
        assert np.abs(v.numpy() - g['sd_' + k]).max() <= 1e-5 * np.abs(g['sd_' + k]).max(), k


def test_reference_checkpoint_loads(golden, tmp_path):
    """A .pt file written by the reference's own save_model (src/models/BaseModel.py:224-236; the checkpoint of the
    run behind tests/golden/run_dccf.npz) loads into the mirrored DCCF through load_model — same keys, same tensors —
    and a checkpoint written here has the reference's keys: the files interchange."""
    g = golden('run_dccf')
    d = synth.write_dataset(str(tmp_path), 'toy', int(g['n_users']), int(g['n_items']), int(g['per_user']), feat_dim=64,
                            seed=int(g['seed']) + 5)
    U, I = g['sd_uid_embeddings.weight'].shape[0], g['sd_iid_embeddings.weight'].shape[0]
    model = _make_model(d, 'toy', U, I, std=0.0)
    from conftest import GOLDEN
    model.load_model(os.path.join(GOLDEN, 'run_dccf_checkpoint.pt'))
    sd = model.state_dict()
    assert sorted(sd) == sorted(k[3:] for k in g.files if k.startswith('sd_'))
    for k, v in sd.items():
        assert np.array_equal(v.numpy(), g['sd_' + k]), k
    model.save_model(str(tmp_path / 'again.pt'))
    again = torch.load(str(tmp_path / 'again.pt'))
    assert sorted(again) == sorted(sd) and all(torch.equal(again[k], sd[k]) for k in sd)


def test_early_stop_and_model_selection_equal_reference():
    """eva_termination / best_result / format_metric on 300 random validation histories (monotone runs, early bests,
    both metric polarities) decided by the unmodified reference (tests/golden/termination.json)."""
    import json
    from conftest import GOLDEN
    cases = json.load(open(os.path.join(GOLDEN, 'termination.json')))
    assert len(cases) >= 300 and any(c['stop'] for c in cases) and not all(c['stop'] for c in cases)
    for c in cases:
        r = BaseRunner(optimizer='Adam', learning_rate=1e-3, metrics=c['metric'] + ',recall@5', dropout=0.0)
        r.valid_results = [list(h) for h in c['history']]
        assert bool(r.eva_termination(None)) == c['stop'], c
        assert utils.best_result(c['metric'], [list(h) for h in c['history']]) == c['best']
        assert utils.format_metric(c['history'][-1]) == c['fmt']


def test_every_cli_flag_equals_reference():
    """All flags of the reference's parsers for the DCCF path (tests/golden/cli_flags.json: option strings, destination,
    default, type — 30-odd flags) exist here with the same spelling, default and type."""
    import json
    from conftest import GOLDEN
    want = json.load(open(os.path.join(GOLDEN, 'cli_flags.json')))
    p = argparse.ArgumentParser()
    utils.parse_global_args(p)
    DataLoader.parse_data_args(p)
    DCCF.parse_model_args(p, model_name='DCCF')
    BaseRunner.parse_runner_args(p)
    DataProcessor.parse_dp_args(p)
    got = {a.dest: a for a in p._actions if a.dest != 'help'}
    assert sorted(got) == sorted(w['dest'] for w in want)
    for w in want:
        a = got[w['dest']]
        assert list(a.option_strings) == w['options'], w
        assert a.default == w['default'], w
        assert getattr(a.type, '__name__', None) == w['type'], w


def test_candidate_layout_contiguous_runs_and_reference_layout():
    """Host side of the ranker call (dccf_b200/models/BaseModel.py::candidate_layout): users whose rows are one
    contiguous run are ranked in place (no index array), the reference's evaluation-set layout — all positives, then
    the blocks of negatives (src/data_processor/DataProcessor.py:92-111) — goes through the grouping index."""
    from dccf_b200.models.BaseModel import candidate_layout, group_candidates
    uid = np.repeat([7, 3, 9, 4], [5, 1, 1001, 2])                    # contiguous, users NOT ascending
    rows, off = candidate_layout(uid)
    assert rows is None and off.tolist() == [0, 5, 6, 1007, 1009]
    rows, off = candidate_layout(np.array([], dtype=np.int64))
    assert rows is None and off.tolist() == [0]
    pos = np.array([1, 1, 2, 5])                                       # positives first, negatives of each user after
    uid = np.concatenate([pos, np.repeat([1, 2, 5], 3)])
    rows, off = candidate_layout(uid)
    users, want_rows, want_off = group_candidates(uid)
    assert rows is not None and np.array_equal(rows, want_rows) and np.array_equal(off, want_off)
    for g, u in enumerate(users):
        assert set(uid[rows[off[g]:off[g + 1]]].tolist()) == {u}
    assert off.tolist() == [0, 5, 9, 13]


def test_n_layers_other_than_one_is_rejected_at_construction():
    """--n_layers is parsed like the reference's (src/models/DMF.py:13-16) but the kernels implement the default single
    Linear(64 + F -> 64): any other depth fails when the model is built, with a message — not at the first predict."""
    import pytest
    from dccf_b200.models.DCCF import DCCF
    with pytest.raises(ValueError, match='n_layers'):
        DCCF(path='', dataset='', sentence_model='', sample_num=2, attribute_num=1, std=0.0, label_min=0, label_max=1,
             feature_num=0, user_num=4, item_num=5, u_vector_size=64, i_vector_size=64, n_layers=2, random_seed=1,
             model_path='/tmp/x.pt', feature_embedding=torch.zeros(5, 64), expo_prob=torch.ones(4, 5))
