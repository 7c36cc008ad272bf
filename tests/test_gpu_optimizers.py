"""GD and Adagrad on the fused training step (dccf_adam.rule 1 / 2) on the GPU: the kernels against the numpy reference
steps, the fused step against the reference's autograd + torch.optim sequence, graph replay, the runner, checkpoints,
the command line and data parallelism."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_err
from test_gpu_parity import make_model, model_params, random_problem
from test_optimizers_cpu import adagrad_step, sgd_step, train_step

pytestmark = pytest.mark.gpu

KINDS = ['gd', 'adagrad']
RULE = {'gd': 1, 'adagrad': 2}
PARAMS = ('E_user', 'E_item', 'W', 'b')
# W: where |g| is tiny, Adagrad's g / sqrt(s) amplifies fp32 summation noise (as Adam's m / sqrt(v) does: see
# EMB_TOL in test_gpu_parity.py)
W_TOL = {'gd': 1e-5, 'adagrad': 5e-4}


def test_fused_step_record_lists_gd_and_adagrad():
    """dccf_adam_step with rules 1 and 2 on the record layout of test_fused_adam_step_record_lists: rows with 1, 2,
    50 and 300 records, and a dense tensor from 20 partials; NULL for the state a rule does not have."""
    from dccf_b200 import kernels
    rs = np.random.RandomState(12)
    rows, n_rec, n_w, n_parts = 700, 900, 5000, 20
    keys = rs.randint(0, rows, size=n_rec).astype(np.int32)
    keys[np.isin(keys, [5, 17, 99])] = 6        # the three rows below get exactly 2, 300 and 50 records
    keys[:300] = 17
    keys[300:350] = 99
    keys[350:352] = 5
    keys = keys[rs.permutation(n_rec)]
    grads = (rs.standard_normal((n_rec, 64)) * 0.01).astype(np.float32)
    table = (rs.standard_normal((rows, 64)) * 0.05).astype(np.float32)
    dense = np.zeros((rows, 64), dtype=np.float32)
    for r in range(n_rec):
        dense[keys[r]] += grads[r]
    Wd = (rs.standard_normal(n_w) * 0.05).astype(np.float32)
    gparts = (rs.standard_normal((n_parts, n_w)) * 0.01).astype(np.float32)
    s0 = (rs.random_sample((rows, 64)) * 1e-4).astype(np.float32)
    sw0 = (rs.random_sample(n_w) * 1e-4).astype(np.float32)
    lens = np.bincount(keys, minlength=rows)
    assert {1, 2, 50, 300} <= set(lens.tolist())
    for kind in KINDS:
        hp = kernels.make_adam(1e-3, 1e-4, 1e-4, step=3, eps=1e-10, rule=RULE[kind])
        t = torch.from_numpy(table).cuda()
        w = torch.from_numpy(Wd).cuda()
        m = torch.from_numpy(s0).cuda() if kind == 'adagrad' else None
        wm = torch.from_numpy(sw0).cuda() if kind == 'adagrad' else None
        head = torch.full((rows,), -1, dtype=torch.int32, device='cuda')
        nxt = torch.empty(n_rec, dtype=torch.int32, device='cuda')
        k_d, g_d, gp_d = torch.from_numpy(keys).cuda(), torch.from_numpy(grads).cuda(), torch.from_numpy(gparts).cuda()
        kernels.adam_step([kernels.adam_table(t, m, None, k_d, g_d, 1, n_rec, n_rec, n_rec * 64, head, nxt)],
                          [kernels.adam_tensor(w, wm, None, gp_d, n_parts, n_w)], hp)
        torch.cuda.synchronize()
        assert int((head != -1).sum()) == 0
        if kind == 'gd':
            want_p, want_W = sgd_step(table, dense, l2=1e-4), sgd_step(Wd, gparts.sum(0))
        else:
            want_p, want_s = adagrad_step(table, dense, s0)
            want_W, want_sw = adagrad_step(Wd, gparts.sum(0), sw0)
            assert rel_err(m.cpu().numpy(), want_s) < 2e-5 and rel_err(wm.cpu().numpy(), want_sw) < 2e-5
        assert rel_err(t.cpu().numpy(), want_p) < 1e-5, kind
        assert rel_err(w.cpu().numpy(), want_W) < 1e-5, kind
        # a rule whose state is missing is refused
        if kind == 'adagrad':
            with pytest.raises(Exception, match='null buffer'):
                kernels.adam_step([kernels.adam_table(t, None, None, k_d, g_d, 1, n_rec, n_rec, n_rec * 64, head, nxt)],
                                  [], hp)


def _check_fused(model, kind, new_params, new_state, tol_w):
    got = model_params(model)
    for k in PARAMS:
        assert rel_err(got[k], new_params[k]) < (tol_w if k == 'W' else 1e-5), (kind, k)
        if kind == 'adagrad':
            assert rel_err(model.optimizer.state_sum[k].cpu().numpy(), new_state[k]['s']) < 2e-5, (kind, k)


def _released(model):
    opt = model.optimizer
    assert int((opt.head_u != -1).sum()) == 0 and int((opt.head_i != -1).sum()) == 0
    if opt.__dict__.get('csr_pool') is not None:
        assert int(opt.csr_pool.abs().sum()) == 0


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('rank', [1, 0])
def test_eager_fused_step_vs_reference_steps(kind, rank):
    """Three eager fused steps with explicit confounders, noise and dropout masks against the numpy reference
    train_step: prediction and loss within 1e-5, tables and b within 1e-5, W within W_TOL, state_sum within 2e-5.
    rank 0: the MSE loss."""
    U, I, F, P, S, A, std, drop = 60, 90, 128, 64, 5, 2, 0.1, 0.2
    params, X, si, noise, mask = random_problem(21, U, I, F, P, S, A, std, drop)
    Y = np.random.RandomState(1).random_sample(P).astype(np.float32) if rank == 0 else None
    model = make_model(params, S, A, std)
    model.optimizer = model.make_fused_optimizer(lr=1e-3, l2=1e-4, kind=kind)
    assert model.optimizer.eps == (1e-10 if kind == 'adagrad' else 1e-8)
    ref = {k: params[k] for k in params}
    state = {k: {'s': np.zeros_like(params[k])} for k in PARAMS}
    hp = dict(lr=1e-3, l2=1e-4, weight_decay=1e-4)
    for t in range(3):
        Xt, sit = np.roll(X, t, axis=0).copy(), np.roll(si, t, axis=0).copy()
        fd = {'X': torch.from_numpy(Xt).cuda(), 'rank': rank, 'train': True, 'dropout': drop,
              'Y': torch.from_numpy(Y).cuda() if Y is not None else torch.zeros(P).cuda(),
              'sample_item': torch.from_numpy(sit), 'noise': torch.from_numpy(noise),
              'dropout_mask': torch.from_numpy(mask)}
        out = model.train_step(fd)
        new, state, loss, pred = train_step(ref, state, t + 1, Xt, sit, noise, mask, A, hp,
                                            loss_mode=0 if rank == 1 else 1, Y=Y, optimizer=kind)
        ref = dict(new, Feat=params['Feat'], expo=params['expo'])
        torch.cuda.synchronize()
        assert abs(float(out['loss']) - loss) < 1e-5 * abs(loss), (t, float(out['loss']), loss)
        assert rel_err(out['prediction'].cpu().numpy(), pred) < 1e-5
        _check_fused(model, kind, ref, state, W_TOL[kind])
        _released(model)
    assert model.optimizer.step_count == 3
    model.check_ids()


@pytest.mark.parametrize('kind', KINDS)
def test_fused_step_is_a_drop_in_for_the_reference_sequence(kind):
    """The fused step against what the reference runs (src/runners/BaseRunner.py:175-188) on the same model and the
    same explicit draws: autograd forward, loss + l2 * model.l2(), backward, clip_grad_value_(50) and
    torch.optim.SGD / Adagrad(weight_decay=l2) — five steps."""
    U, I, F, P, S, A, std, drop = 60, 90, 128, 64, 5, 2, 0.1, 0.2
    lr, l2 = 1e-2, 1e-4
    params, X, si, noise, mask = random_problem(23, U, I, F, P, S, A, std, drop)
    fused = make_model(params, S, A, std)
    fused.optimizer = fused.make_fused_optimizer(lr=lr, l2=l2, weight_decay=l2, kind=kind)
    ref = make_model(params, S, A, std)
    assert len(list(ref.parameters())) == 4
    opt = torch.optim.SGD(ref.parameters(), lr=lr, weight_decay=l2) if kind == 'gd' else \
        torch.optim.Adagrad(ref.parameters(), lr=lr, weight_decay=l2)
    for t in range(5):
        Xt, sit = np.roll(X, 3 * t, axis=0).copy(), np.roll(si, t, axis=0).copy()

        def fd():
            return {'X': torch.from_numpy(Xt).cuda(), 'rank': 1, 'train': True, 'dropout': drop, 'Y': torch.zeros(P).cuda(),
                    'sample_item': torch.from_numpy(sit), 'noise': torch.from_numpy(noise),
                    'dropout_mask': torch.from_numpy(mask)}
        out_f = fused.train_step(fd())
        ref.train()
        opt.zero_grad()
        out_r = ref(fd())
        loss = out_r['loss'] + ref.l2() * l2
        loss.backward()
        torch.nn.utils.clip_grad_value_(ref.parameters(), 50)
        opt.step()
        torch.cuda.synchronize()
        assert abs(float(out_f['loss']) - float(out_r['loss'])) < 1e-5 * abs(float(out_r['loss'])), t
        assert rel_err(out_f['prediction'].cpu().numpy(), out_r['prediction'].detach().cpu().numpy()) < 1e-5
        got, want = model_params(fused), model_params(ref)
        for k in PARAMS:
            assert rel_err(got[k], want[k]) < (W_TOL[kind] if k == 'W' else 1e-5), (t, k)
        if kind == 'adagrad':
            pmap = dict(zip(PARAMS, (ref.uid_embeddings.weight, ref.iid_embeddings.weight, ref.mlp[0].weight,
                                     ref.mlp[0].bias)))
            for k, p in pmap.items():
                assert rel_err(fused.optimizer.state_sum[k].cpu().numpy(), opt.state[p]['sum'].cpu().numpy()) < 2e-5, k


@pytest.mark.parametrize('kind', KINDS)
def test_graph_replay_equals_eager_steps(kind):
    """CUDA-graph replay of the GD / Adagrad step is bit-identical to launching its kernels one by one."""
    U, I, F, P, S, A, std, drop = 200, 300, 768, 64, 10, 2, 0.1, 0.2
    params, X, si, _, _ = random_problem(8, U, I, F, P, S, A, 0.0, 0.0)
    outs = []
    for use_graph in (False, True):
        model = make_model(params, S, A, std)
        model.use_cuda_graph = use_graph
        model.optimizer = model.make_fused_optimizer(lr=1e-3, l2=1e-4, kind=kind)
        losses = []
        for t in range(6):
            Xt = np.roll(X, t, axis=0).copy()
            Xt[P // 2:, 0] = Xt[:P // 2, 0]
            fd = {'X': torch.from_numpy(Xt).cuda(), 'rank': 1, 'train': True, 'dropout': drop,
                  'Y': torch.zeros(P).cuda(), 'sample_item': torch.from_numpy(np.roll(si, t, axis=0).copy())}
            losses.append(float(model.train_step(fd)['loss']))
        state = {k: v.cpu().numpy() for k, v in getattr(model.optimizer, 'state_sum', {}).items()}
        outs.append((losses, model_params(model), state, model.optimizer.step_count))
    assert outs[0][0] == outs[1][0]
    assert outs[0][3] == outs[1][3] == 6
    for k in PARAMS:
        assert np.array_equal(outs[0][1][k], outs[1][1][k]), k
    for k in outs[0][2]:
        assert np.array_equal(outs[0][2][k], outs[1][2][k]), k
    assert (len(outs[0][2]) == 4) == (kind == 'adagrad')


def _toy(tmp_path):
    """(datasets root, dataset directory) of the toy dataset the command-line tests use."""
    from dccf_b200 import synth
    data_root = str(tmp_path / 'datasets')
    d = synth.write_dataset(data_root, 'toy', n_users=300, n_items=400, per_user=12, feat_dim=768, seed=1)
    return data_root, d


@pytest.mark.parametrize('name,kind', [('GD', 'gd'), ('Adagrad', 'adagrad')])
def test_runner_fits_with_the_fused_gd_and_adagrad_step(tmp_path, name, kind):
    """BaseRunner(optimizer='GD' / 'Adagrad').fit takes the device-resident epoch of the fused step: the optimizer is
    the fused state, not a torch Optimizer, and the parameters move."""
    from dccf_b200 import synth
    from dccf_b200.data_loaders.DataLoader import DataLoader
    from dccf_b200.data_processor.DataProcessor import DataProcessor
    from dccf_b200.models.DCCF import DCCF, FusedAdamState
    from dccf_b200.runners.BaseRunner import BaseRunner
    data_root, d = _toy(tmp_path)
    torch.manual_seed(3)
    np.random.seed(3)
    dl = DataLoader(path=data_root, dataset='toy', label='label', sep=',')
    model = DCCF(path=d, dataset='toy', sentence_model=synth.DEFAULT_SENTENCE_MODEL,
                 sample_num=10, attribute_num=2, std=0.1, label_min=0, label_max=1, feature_num=0,
                 user_num=dl.user_num, item_num=dl.item_num, u_vector_size=64, i_vector_size=64, n_layers=1,
                 random_seed=3, model_path=str(tmp_path / 'm.pt'))
    model.apply(model.init_paras)
    model = model.cuda()
    dl.drop_neg()
    dp = DataProcessor(dl, model, rank=1, test_neg_n=100)
    dp.get_test_data()
    dp.get_validation_data()
    before = {k: v.copy() for k, v in model_params(model).items()}
    resident = []
    begin = model.begin_resident_epoch

    def counted(*a, **kw):
        resident.append(1)
        return begin(*a, **kw)
    model.begin_resident_epoch = counted
    runner = BaseRunner(optimizer=name, learning_rate=0.01, l2=1e-4, batch_size=32, metrics='ndcg@5')
    runner.show_progress = False
    dp.get_train_data(epoch=-1)
    out = runner.fit(model, dp.get_train_data(epoch=0), dp, epoch=0)
    torch.cuda.synchronize()
    assert resident, 'the device-resident epoch was not used'
    assert isinstance(model.optimizer, FusedAdamState) and model.optimizer.kind == kind
    assert not isinstance(model.optimizer, torch.optim.Optimizer)
    assert model.optimizer.step_count > 2 and np.isfinite(float(out['loss']))
    after = model_params(model)
    for k in PARAMS:
        assert np.isfinite(after[k]).all() and not np.array_equal(after[k], before[k]), k
    _released(model)


def test_adagrad_checkpoint_resume_is_bit_identical(tmp_path):
    """save_training_state / load_training_state with Adagrad (weights, state_sum, step, stream position): the resumed
    run equals the uninterrupted one bit for bit.  Loading it into a fused optimizer of another kind is refused."""
    U, I, F, P, S, A = 120, 150, 128, 32, 10, 2
    params, X, si, _, _ = random_problem(31, U, I, F, P, S, A, 0.0, 0.0)
    X[P // 2:, 0] = X[:P // 2, 0]

    def steps(model, t0, t1):
        out = []
        for t in range(t0, t1):
            o = model.train_step({'X': torch.from_numpy(X).cuda(), 'rank': 1, 'train': True, 'dropout': 0.2,
                                  'Y': torch.zeros(P).cuda(), 'sample_item': torch.from_numpy(np.roll(si, t, axis=0).copy())})
            out.append(float(o['loss']))
        return out

    a = make_model(params, S, A, 0.1)
    a.optimizer = a.make_fused_optimizer(lr=1e-2, l2=1e-4, kind='adagrad')
    steps(a, 0, 3)
    path = a.save_training_state(str(tmp_path / 'run.train_state'))
    la = steps(a, 3, 6)
    b = make_model(params, S, A, 0.1)
    b.load_training_state(path)
    assert b.optimizer.kind == 'adagrad' and b.optimizer.step_count == 3
    lb = steps(b, 3, 6)
    assert la == lb
    pa, pb = model_params(a), model_params(b)
    for k in PARAMS:
        assert np.array_equal(pa[k], pb[k]), k
        assert torch.equal(a.optimizer.state_sum[k], b.optimizer.state_sum[k]), k
    c = make_model(params, S, A, 0.1)
    c.optimizer = c.make_fused_optimizer(lr=1e-2, l2=1e-4, kind='gd')
    with pytest.raises(ValueError, match='adagrad'):
        c.load_training_state(path)


@pytest.mark.parametrize('optimizer', [None, 'Adagrad'])
def test_main_cli_trains_with_gd_and_adagrad(tmp_path, optimizer):
    """src/main.py --model_name DCCF without --optimizer (the reference's default, GD) and with --optimizer Adagrad."""
    data_root, _ = _toy(tmp_path)
    cmd = [sys.executable, 'main.py', '--rank', '1', '--model_name', 'DCCF', '--lr', '0.01',
           '--dataset', 'toy', '--path', data_root + '/', '--metric', 'ndcg@5,recall@5', '--gpu', '0',
           '--epoch', '2', '--test_neg_n', '100', '--log_file', str(tmp_path / 'log.txt'),
           '--result_file', str(tmp_path / 'result.npy'), '--model_path', str(tmp_path / 'model' / 'm.pt')]
    if optimizer is not None:
        cmd += ['--optimizer', optimizer]
    r = subprocess.run(cmd, cwd=os.path.join(ROOT, 'src'), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    log = open(str(tmp_path / 'log.txt')).read()
    assert 'Optimizer: %s' % (optimizer or 'GD') in log
    assert 'Test After Training' in log and 'Epoch     2' in log
    assert np.isfinite(np.load(str(tmp_path / 'result.npy'))).all()


@pytest.mark.parametrize('kind', KINDS)
def test_data_parallel_gd_and_adagrad_equal_single_gpu(kind):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29523', os.path.join(ROOT, 'tools', 'dp_check.py'),
           '--optimizer', kind]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0 and 'DP CHECK OK' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
