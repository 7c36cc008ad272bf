"""Rating prediction (--rank 0, MSE loss) on the device-resident epoch and data parallel, on the GPU: the resident epoch
against the step-by-step run, the runner, the staged labels, the kernel count of a step, the global MSE divisor of a
data-parallel step, and (with two GPUs) the data-parallel check and the command line under torchrun."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from test_gpu_parity import make_model, model_params, random_problem

pytestmark = pytest.mark.gpu

KINDS = ['adam', 'gd', 'adagrad']
PARAMS = ('E_user', 'E_item', 'W', 'b')
STATE = {'adam': ('exp_avg', 'exp_avg_sq'), 'gd': (), 'adagrad': ('state_sum',)}


def _epoch(n, P, I, seed):
    """n batches of P rating pairs and their labels, plus a ragged last batch of P // 2 + 3 pairs."""
    rs = np.random.RandomState(seed)
    Xs = np.stack([rs.randint(0, 200, size=P), rs.randint(0, I, size=P)], 1)
    Xs = np.stack([np.roll(Xs, 3 * t, axis=0) for t in range(n)]).astype(np.int64)
    Ys = rs.uniform(1.0, 5.0, size=(n, P)).astype(np.float32)
    Pt = P // 2 + 3
    Xt = np.stack([rs.randint(0, 200, size=Pt), rs.randint(0, I, size=Pt)], 1).astype(np.int64)
    Yt = rs.uniform(1.0, 5.0, size=Pt).astype(np.float32)
    return Xs, Ys, Xt, Yt


def _opt_state(opt):
    return {n + ' ' + k: t.cpu().numpy() for n in STATE[opt.kind] for k, t in getattr(opt, n).items()}


@pytest.mark.parametrize('kind', KINDS)
def test_rank0_resident_epoch_equals_step_by_step(kind):
    """A rank-0 resident epoch (labels staged by the step's first kernel) and a ragged last batch are bit-identical to
    the same batches fed one by one through train_step: per-step predictions and losses, final parameters, optimizer
    state and the CPU generator's position."""
    U, I, F, P, S, A, std, drop = 200, 300, 768, 64, 10, 2, 0.1, 0.2
    params, _, _, _, _ = random_problem(8, U, I, F, P, S, A, 0.0, 0.0)
    n = 5
    Xs, Ys, Xt, Yt = _epoch(n, P, I, 21)
    outs = []
    for resident in (False, True):
        model = make_model(params, S, A, std)
        model.optimizer = model.make_fused_optimizer(lr=1e-3, l2=1e-4, kind=kind)
        torch.manual_seed(4242)
        preds, losses = [], []
        if resident:
            draws = model.draw_confounders(n * P).view(n, P, S)
            step = model.begin_resident_epoch(torch.from_numpy(Xs).cuda(), draws.cuda(), drop,
                                              Y_epoch=torch.from_numpy(Ys).cuda())
            preds.append(step.first['prediction'].cpu().numpy())
            losses.append(float(step.first['loss']))
            while step.remaining() > 0:
                o = step()
                preds.append(o['prediction'].cpu().numpy())
                losses.append(float(o['loss']))
            assert len(losses) == n
        else:
            for t in range(n):
                o = model.train_step({'X': torch.from_numpy(Xs[t]).cuda(), 'rank': 0, 'train': True, 'dropout': drop,
                                      'Y': torch.from_numpy(Ys[t]).cuda()})
                preds.append(o['prediction'].cpu().numpy())
                losses.append(float(o['loss']))
        o = model.train_step({'X': torch.from_numpy(Xt).cuda(), 'rank': 0, 'train': True, 'dropout': drop,
                              'Y': torch.from_numpy(Yt).cuda()})
        preds.append(o['prediction'].cpu().numpy())
        losses.append(float(o['loss']))
        torch.cuda.synchronize()
        outs.append((preds, losses, model_params(model), _opt_state(model.optimizer), model.optimizer.step_count,
                     torch.randint(1000, (3,)).numpy()))
    (p0, l0, w0, s0, c0, g0), (p1, l1, w1, s1, c1, g1) = outs
    assert l0 == l1 and all(np.isfinite(l0))
    assert len(p0) == len(p1) == n + 1
    for a, b in zip(p0, p1):
        assert np.array_equal(a, b)
    assert c0 == c1 == n + 1 and np.array_equal(g0, g1)
    for k in PARAMS:
        assert np.array_equal(w0[k], w1[k]), k
    assert sorted(s0) == sorted(s1) and len(s0) == 4 * len(STATE[kind])
    for k in s0:
        assert np.array_equal(s0[k], s1[k]), k


def test_staged_labels_and_kernel_count():
    """The labels the step's first kernel stages for step k are Y_epoch[k]; a rank-0 resident step is a graph of as
    many kernels as a rank-1 one.  dccf_stage_batch (the staging launch of configurations without the split step)
    copies the labels of batch *cursor as well."""
    from dccf_b200 import kernels
    U, I, F, P, S, A, std, drop = 200, 300, 768, 64, 10, 2, 0.1, 0.2
    params, _, _, _, _ = random_problem(9, U, I, F, P, S, A, 0.0, 0.0)
    n = 4
    Xs, Ys, _, _ = _epoch(n, P, I, 5)
    X_dev, Y_dev = torch.from_numpy(Xs).cuda(), torch.from_numpy(Ys).cuda()
    model = make_model(params, S, A, std)
    model.optimizer = opt = model.make_fused_optimizer(lr=1e-3, l2=1e-4)
    draws = model.draw_confounders(n * P).view(n, P, S).cuda()
    step = model.begin_resident_epoch(X_dev, draws, drop, Y_epoch=Y_dev)
    g0 = model._graphs[(P, 0, drop, opt, True, False)]
    k = 1
    while step.remaining() > 0:
        step()
        torch.cuda.synchronize()
        assert torch.equal(g0['Y'], Y_dev[k]), k
        assert torch.equal(g0['X'], X_dev[k]) and torch.equal(g0['si'], draws[k]), k
        k += 1
    assert k == n
    # the BPR epoch of the same shape on the same model
    Xb = X_dev.clone()
    Xb[:, P // 2:, 0] = Xb[:, :P // 2, 0]
    step = model.begin_resident_epoch(Xb, draws, drop)
    while step.remaining() > 0:
        step()
    g1 = model._graphs[(P, 1, drop, opt, True, False)]
    assert g0['n_kernels'] == g1['n_kernels'] > 0

    ptrs = torch.tensor([X_dev.data_ptr(), draws.data_ptr(), 0, 0, 0, 0, Y_dev.data_ptr()], dtype=torch.int64).cuda()
    cursor = torch.full((1,), 2, dtype=torch.int64, device='cuda')
    X_out = torch.zeros((P, 2), dtype=torch.int64, device='cuda')
    si_out = torch.zeros((P, S), dtype=torch.int64, device='cuda')
    Y_out = torch.zeros(P, dtype=torch.float32, device='cuda')
    kernels.stage_batch(ptrs, cursor, P, S, X_out, si_out, Y_out)
    torch.cuda.synchronize()
    assert torch.equal(X_out, X_dev[2]) and torch.equal(si_out, draws[2]) and torch.equal(Y_out, Y_dev[2])
    assert int(cursor) == 3


def test_global_mse_divisor_halves_gradients_and_loss():
    """The MSE pair count of a data-parallel step, on one GPU: with a count of 2P every gradient record, every dW / db
    partial and the loss are exactly half of those of the count = P call (scaling by a power of two is exact), and the
    predictions are unchanged."""
    from dccf_b200 import kernels
    U, I, F, P, S, A, std, drop = 200, 300, 768, 96, 10, 2, 0.1, 0.2
    params, X, si, noise, mask = random_problem(14, U, I, F, P, S, A, std, drop)
    model = make_model(params, S, A, std)
    Y = torch.from_numpy(np.random.RandomState(2).uniform(1, 5, P).astype(np.float32)).cuda()
    call = model._make_call({'X': torch.from_numpy(X).cuda(), 'sample_item': torch.from_numpy(si),
                             'noise': torch.from_numpy(noise), 'dropout_mask': torch.from_numpy(mask), 'dropout': drop})
    N = call['N']

    def run(mse_pairs):
        rec = model._rec_buffers(call, 1, kernels.train_bwd_splits(N, F))
        pred = torch.empty(P, dtype=torch.float32, device='cuda')
        ws = lambda shape: torch.empty(shape, dtype=torch.float32, device='cuda')    # noqa: E731
        kernels.train_fwd_bwd_tc(
            model._dims(), model.uid_embeddings.weight.data, model.iid_embeddings.weight.data, model.feature_embedding,
            model.mlp[0].weight.data, model.mlp[0].bias.data, model._expo(), call['X'], call['sample_item'], Y,
            call['rng'], 1, pred, rec['loss'], ws(kernels.train_w_image_floats(F)), False,
            ws((kernels.train_fwd_ksplits(N, F), N, 64)), ws((N, 64)), ws(P), rec['gW_part'], rec['gb_part'],
            rec['gu_rec'], rec['gi_rec'], rec['keys_u'], rec['keys_i'], err_flag=model._err_flag, mse_pairs=mse_pairs)
        torch.cuda.synchronize()
        return {k: rec[k].clone() for k in ('loss', 'gW_part', 'gb_part', 'gu_rec', 'gi_rec', 'keys_u', 'keys_i')}, pred

    one, pred1 = run(0)
    same, _ = run(P)
    two, pred2 = run(2 * P)
    assert torch.equal(pred1, pred2)
    for k in one:
        assert torch.equal(one[k], same[k]), k
    for k in ('keys_u', 'keys_i'):
        assert torch.equal(one[k], two[k]), k
    for k in ('loss', 'gW_part', 'gb_part', 'gu_rec', 'gi_rec'):
        assert torch.equal(two[k] * 2, one[k]), k
    assert float(one['loss']) > 0
    model.check_ids()


def test_runner_fit_rank0_takes_the_resident_epoch_and_equals_step_by_step(tmp_path):
    """BaseRunner.fit on a --rank 0 data processor takes the device-resident epoch (counted) and ends bit-identical to
    _fit_remaining, the step-by-step loop, over the same batches: parameters, Adam state, the last batch's loss."""
    from dccf_b200 import synth
    from dccf_b200.data_loaders.DataLoader import DataLoader
    from dccf_b200.data_processor.DataProcessor import DataProcessor
    from dccf_b200.models.DCCF import DCCF
    from dccf_b200.runners.BaseRunner import BaseRunner
    data_root = str(tmp_path / 'datasets')
    d = synth.write_dataset(data_root, 'toy', n_users=300, n_items=400, per_user=12, feat_dim=768, seed=1)
    res = []
    for resident in (True, False):
        torch.manual_seed(3)
        np.random.seed(3)
        dl = DataLoader(path=data_root, dataset='toy', label='label', sep=',')
        model = DCCF(path=d, dataset='toy', sentence_model=synth.DEFAULT_SENTENCE_MODEL, sample_num=10,
                     attribute_num=2, std=0.1, label_min=0, label_max=1, feature_num=0, user_num=dl.user_num,
                     item_num=dl.item_num, u_vector_size=64, i_vector_size=64, n_layers=1, random_seed=3,
                     model_path=str(tmp_path / 'm.pt'))
        model.apply(model.init_paras)
        model = model.cuda()
        dp = DataProcessor(dl, model, rank=0, test_neg_n=100)
        calls = []
        begin = model.begin_resident_epoch

        def counted(*a, **kw):
            calls.append(kw.get('Y_epoch') is not None)
            return begin(*a, **kw)
        model.begin_resident_epoch = counted
        runner = BaseRunner(optimizer='Adam', learning_rate=0.01, l2=1e-4, batch_size=32, metrics='rmse')
        runner.show_progress = False
        data = dp.get_train_data(epoch=0)
        torch.manual_seed(11)
        if resident:
            out = runner.fit(model, data, dp, epoch=0)
            assert calls and all(calls), 'the rank-0 device-resident epoch was not used'
        else:
            model.optimizer = runner._build_optimizer(model)
            batches = runner.batches_add_control(dp.prepare_batches(data, runner.batch_size, train=True), train=True)
            assert len(batches) > 2
            model.train()
            out = runner._fit_remaining(model, batches, True, runner.batch_size, 0, None)
            model.eval()
            assert not calls
        torch.cuda.synchronize()
        res.append((float(out['loss']), out['prediction'].cpu().numpy(), model_params(model),
                    _opt_state(model.optimizer), model.optimizer.step_count))
    (l0, p0, w0, s0, c0), (l1, p1, w1, s1, c1) = res
    assert l0 == l1 and np.isfinite(l0) and np.array_equal(p0, p1) and c0 == c1 > 2
    for k in PARAMS:
        assert np.array_equal(w0[k], w1[k]), k
    for k in s0:
        assert np.array_equal(s0[k], s1[k]), k


@pytest.mark.parametrize('kind', KINDS)
def test_data_parallel_rank0_equals_single_gpu(kind):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29527', os.path.join(ROOT, 'tools', 'dp_check.py'),
           '--optimizer', kind, '--rank', '0']
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0 and 'DP CHECK OK' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_cli_data_parallel_rank0_training(tmp_path):
    """src/main.py --rank 0 under torchrun on 2 GPUs: trains, evaluates RMSE / MAE user-sharded, writes its files and
    ends with identical parameter checksums on both ranks."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    from dccf_b200 import synth
    data_root = str(tmp_path / 'datasets')
    synth.write_dataset(data_root, 'toy', n_users=300, n_items=400, per_user=12, feat_dim=768, seed=1)
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', '29529', 'main.py', '--rank', '0', '--model_name', 'DCCF', '--optimizer', 'Adam',
           '--lr', '0.001', '--dataset', 'toy', '--path', data_root + '/', '--metric', 'rmse,mae',
           '--epoch', '2', '--batch_size', '32', '--log_file', str(tmp_path / 'log.txt'),
           '--result_file', str(tmp_path / 'result.npy'), '--model_path', str(tmp_path / 'model' / 'm.pt')]
    r = subprocess.run(cmd, cwd=os.path.join(ROOT, 'src'), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    log = open(str(tmp_path / 'log.txt')).read()
    assert 'data parallel: 2 ranks' in log and 'parameter checksums identical on all 2 ranks' in log
    assert 'Test After Training' in log and 'Epoch     2' in log
    assert os.path.exists(str(tmp_path / 'result.npy')) and os.path.exists(str(tmp_path / 'model' / 'm.pt'))
