"""BiasedMF / IPSBiasedMF on the GPU: predictions and the exported exposure matrix against the reference
(tests/golden/ipsmf.npz), one training step against the float64 trainer (tests/mf_reference.py) element by element,
determinism of graph replay and of device-resident epochs, the id check, 20 steps of drift, and the end-to-end path
main.py IPSBiasedMF -> tools/export_exposure.py -> main.py DCCF."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import rel_err
from mf_reference import forward, init_state, step

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# Per-element bound of the one-step comparison: C * 2^-20 * (first-order magnitude of the element) + 1 ulp.  C is about
# 5x the largest value the kernels needed: 0.203 (E_item), on an NVIDIA B200 at a 1000 W power limit.
C = 1.0
UNIT = C * 2.0 ** -20
NAMES = {'E_user': 'uid_embeddings.weight', 'E_item': 'iid_embeddings.weight', 'user_bias': 'user_bias.weight',
         'item_bias': 'item_bias.weight', 'global_bias': 'global_bias'}


def make_model(U, I, seed=2019, prop=None, M=0.1, scale=10.0, cls='IPSBiasedMF'):
    from dccf_b200.models.BiasedMF import BiasedMF
    from dccf_b200.models.IPSBiasedMF import IPSBiasedMF
    common = dict(label_min=0, label_max=1, feature_num=0, user_num=U, item_num=I, u_vector_size=64, i_vector_size=64,
                  random_seed=seed, model_path='/tmp/unused_mf.pt')
    if cls == 'IPSBiasedMF':
        if prop is None:
            prop = np.random.RandomState(seed).random_sample(I).astype(np.float32)
        model = IPSBiasedMF(path='', dataset='', M=M, propensity=prop, **common)
    else:
        model = BiasedMF(**common)
    model.apply(model.init_paras)
    with torch.no_grad():           # predictions of order 1: every term of the step counts
        for p in model.parameters():
            p.mul_(scale)
    return model.cuda()


def host_params(model):
    sd = model.state_dict()
    out = {k: sd[v].detach().double().cpu().numpy().copy() for k, v in NAMES.items()}
    out['user_bias'], out['item_bias'] = out['user_bias'].reshape(-1), out['item_bias'].reshape(-1)
    return out


def batch(rs, U, I, P, rank):
    X = np.stack([rs.randint(0, U, P), rs.randint(0, I, P)], 1).astype(np.int64)
    if rank == 1:
        X[P // 2:, 0] = X[:P // 2, 0]
        Y = np.r_[np.ones(P // 2), np.zeros(P // 2)].astype(np.float32)
    else:
        Y = rs.randint(1, 6, P).astype(np.float32)
    return X, Y


def feed(X, Y, rank):
    return {'X': torch.from_numpy(X).cuda(), 'Y': torch.from_numpy(Y).cuda(), 'rank': rank, 'train': True,
            'dropout': 0.0}


def ulp(x):
    return np.spacing(np.abs(np.asarray(x, np.float32))).astype(np.float64)


def check(name, got, want, bound):
    got = np.asarray(got, np.float64).reshape(np.shape(want))
    err = np.abs(got - want)
    ok = err <= bound
    need = float(np.max((err - ulp(want)).clip(0) / np.maximum(bound - ulp(want), 1e-300) * C))
    print('%-22s max needed C %.3f' % (name, need))
    assert ok.all(), '%s: %d elements out of bound, worst %g vs %g' % (
        name, int((~ok).sum()), float(err.ravel()[np.argmax(err - bound)]), float(bound.ravel()[np.argmax(err - bound)]))


def test_predict_and_export_match_reference(golden, tmp_path):
    g = golden('ipsmf')
    U, I = g['pred'].shape
    model = make_model(U, I, prop=g['propensity'], M=float(g['mf_min_propensity']), scale=1.0)
    with torch.no_grad():
        model.uid_embeddings.weight.copy_(torch.from_numpy(g['mf_user']))
        model.iid_embeddings.weight.copy_(torch.from_numpy(g['mf_item']))
        model.user_bias.weight.copy_(torch.from_numpy(g['mf_user_bias']).view(-1, 1))
        model.item_bias.weight.copy_(torch.from_numpy(g['mf_item_bias']).view(-1, 1))
        model.global_bias.fill_(float(g['mf_global_bias']))
    uu, ii = np.meshgrid(np.arange(U), np.arange(I), indexing='ij')
    X = np.stack([uu.reshape(-1), ii.reshape(-1)], 1).astype(np.int64)
    pred = model.predict({'X': torch.from_numpy(X).cuda()})['prediction'].cpu().numpy().reshape(U, I)
    assert rel_err(pred, g['pred']) < 1e-5
    model.check_ids()
    # the export tool on a checkpoint of the same model, in blocks that do not divide U
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    try:
        import export_exposure
    finally:
        sys.path.remove(os.path.join(ROOT, 'tools'))
    d = tmp_path / 'ds'
    d.mkdir()
    np.save(str(d / 'ds.propensity.npy'), g['propensity'])
    model.save_model(str(tmp_path / 'm.pt'))
    mat, npz = export_exposure.export(str(tmp_path), 'ds', str(tmp_path / 'm.pt'), M=float(g['mf_min_propensity']),
                                      block_users=17)
    assert rel_err(np.load(mat), g['pred']) < 1e-5
    f = np.load(npz)
    from dccf_b200 import synth
    assert sorted(f.files) == sorted(synth.make_ipsmf_factors(2, 2))
    assert np.array_equal(f['mf_user'], g['mf_user']) and float(f['mf_global_bias']) == float(g['mf_global_bias'])


@pytest.mark.parametrize('kind', ['adam', 'gd', 'adagrad'])
@pytest.mark.parametrize('rank', [1, 0])
def test_one_step_matches_float64_trainer(kind, rank):
    """Every row of both tables (touched ones with several records, untouched ones), both bias vectors, global_bias,
    the optimizer state and the loss of one eager step."""
    U, I, P = 50, 70, 256
    prop = np.random.RandomState(1).random_sample(I).astype(np.float32)
    prop[:3] = [0.0, 0.05, 0.1]                                 # below and at the clamp M
    model = make_model(U, I, prop=prop, M=0.1)
    hp = {'lr': 1e-2, 'l2': 1e-4, 'weight_decay': 1e-4}
    opt = model.optimizer = model.make_fused_optimizer(lr=hp['lr'], l2=hp['l2'], kind=kind)
    X, Y = batch(np.random.RandomState(2), U, I, P, rank)
    p0 = host_params(model)
    out = model.train_step(feed(X, Y, rank))
    torch.cuda.synchronize()
    model.check_ids()
    p1, s1, loss, pred, info = step(p0, init_state(p0, kind), 1, X, Y, rank, hp, kind, prop=prop, M=0.1)
    got = host_params(model)
    eps = {'adam': 1e-8, 'adagrad': 1e-10}.get(kind)
    for k in p0:
        g, dg = info['g'][k], UNIT * info['mag'][k]
        if kind == 'gd':
            bound = hp['lr'] * dg
        else:
            bound = hp['lr'] * dg * eps / (np.abs(g) + eps) ** 2 + UNIT * np.abs(p1[k] - p0[k])
        check(k, got[k], p1[k], bound + ulp(p1[k]))
        st = opt.state_dict()
        if kind == 'adam':
            check(k + ' exp_avg', st['exp_avg'][k].cpu().numpy(), s1[k]['m'], 0.1 * dg + ulp(s1[k]['m']))
            check(k + ' exp_avg_sq', st['exp_avg_sq'][k].cpu().numpy(), s1[k]['v'],
                  0.001 * 2 * np.abs(g) * dg + UNIT * s1[k]['v'] + ulp(s1[k]['v']))
        elif kind == 'adagrad':
            check(k + ' state_sum', st['state_sum'][k].cpu().numpy(), s1[k]['s'],
                  2 * np.abs(g) * dg + UNIT * s1[k]['s'] + ulp(s1[k]['s']))
    check('loss', out['loss'].cpu().numpy(), np.asarray(loss), np.asarray(UNIT * info['loss_mag'] + ulp(loss)))
    pmag = forward(p0, X, prop, 0.1)[2]
    check('prediction', out['prediction'].cpu().numpy(), pred, UNIT * pmag + ulp(pred))


def _train(model, opt, batches, rank):
    for X, Y in batches:
        model.train_step(feed(X, Y, rank), opt)
    torch.cuda.synchronize()
    return host_params(model), {k: v.clone() for k, v in opt.state_dict().get('exp_avg', {}).items()}


@pytest.mark.parametrize('rank', [1, 0])
def test_graph_replay_equals_eager_and_runs_repeat(rank):
    U, I, P = 300, 500, 128
    rs = np.random.RandomState(4)
    batches = [batch(rs, U, I, P, rank) for _ in range(6)]
    results = []
    for graph in (False, True, True):
        model = make_model(U, I)
        model.use_cuda_graph = graph
        opt = model.optimizer = model.make_fused_optimizer(lr=1e-2, l2=1e-4)
        results.append(_train(model, opt, batches, rank))
        if graph:
            assert any(isinstance(v, dict) for v in model._graphs.values())      # the replays did run
    for other in results[1:]:
        for k in results[0][0]:
            assert np.array_equal(results[0][0][k], other[0][k]), k
        for k in results[0][1]:
            assert torch.equal(results[0][1][k], other[1][k]), k


@pytest.mark.parametrize('rank', [1, 0])
def test_resident_epoch_with_ragged_tail_equals_step_loop(rank):
    """BaseRunner.fit's device-resident epoch (one graph replay per batch, batch staged through the cursor) followed by
    the ragged last batch == the same batches one eager step at a time."""
    from dccf_b200.runners.BaseRunner import BaseRunner
    U, I, P = 300, 500, 64
    rs = np.random.RandomState(5)
    full = [batch(rs, U, I, P, rank) for _ in range(7)]
    tail = batch(rs, U, I, 40, rank)
    ref = make_model(U, I)
    ref.use_cuda_graph = False
    opt = ref.optimizer = ref.make_fused_optimizer(lr=1e-2, l2=1e-4, kind='adagrad')
    want = _train(ref, opt, full + [tail], rank)[0]
    model = make_model(U, I)
    runner = BaseRunner(optimizer='Adagrad', learning_rate=1e-2, l2=1e-4, batch_size=P // 2 if rank == 1 else P)
    runner.show_progress = False

    class DP(object):          # the two things fit asks of a data processor
        def __init__(self):
            self.rank = rank

        def prepare_batches(self, data, batch_size, train):
            return [{'X': torch.from_numpy(X).cuda(), 'Y': torch.from_numpy(Y).cuda(), 'rank': rank}
                    for X, Y in full + [tail]]

    runner.fit(model, None, DP())
    torch.cuda.synchronize()
    got = host_params(model)
    assert model.optimizer.step_count == len(full) + 1
    assert any(k[3] for k, v in model._graphs.items() if isinstance(v, dict))       # the resident graph ran
    for k in want:
        assert np.array_equal(got[k], want[k]), k


def test_out_of_range_ids_raise_the_flag():
    U, I = 20, 30
    model = make_model(U, I)
    model.optimizer = model.make_fused_optimizer(lr=1e-2, l2=1e-4)
    X, Y = batch(np.random.RandomState(6), U, I, 16, 1)
    X[3, 0] = U + 4
    model.train_step(feed(X, Y, 1))
    with pytest.raises(IndexError):
        model.check_ids()
    model.check_ids()                       # cleared
    X[3, 0], X[5, 1] = 0, -1
    model.predict({'X': torch.from_numpy(X).cuda()})
    with pytest.raises(IndexError):
        model.check_ids()


def test_twenty_steps_stay_close_to_float64_trainer():
    U, I, P = 200, 300, 256
    model = make_model(U, I)
    hp = {'lr': 1e-2, 'l2': 1e-4, 'weight_decay': 1e-4}
    model.optimizer = model.make_fused_optimizer(lr=hp['lr'], l2=hp['l2'], kind='adam')
    params = host_params(model)
    state = init_state(params, 'adam')
    prop = model.propensity.cpu().numpy()
    rs = np.random.RandomState(7)
    for t in range(1, 21):
        X, Y = batch(rs, U, I, P, 1)
        out = model.train_step(feed(X, Y, 1))
        params, state, loss, _, _ = step(params, state, t, X, Y, 1, hp, 'adam', prop=prop, M=0.1)
        assert abs(float(out['loss']) - loss) <= 1e-4 * abs(loss)
    got = host_params(model)
    for k in params:
        assert rel_err(got[k], params[k]) < 2e-5, k


def test_end_to_end_train_export_then_dccf(tmp_path):
    """main.py --model_name IPSBiasedMF (2 epochs) -> tools/export_exposure.py -> main.py --model_name DCCF (1 epoch) on
    the exported matrix; the dense file and the factor file give DCCF the same exposure."""
    from dccf_b200 import synth
    U, I, per = synth.PRESETS['tiny']
    synth.write_dataset(str(tmp_path), 'tiny', U, I, per, ipsmf=True)
    os.remove(str(tmp_path / 'tiny' / 'tiny.ips_expo_prob.npy'))        # DCCF must read the exported one
    ckpt = str(tmp_path / 'mf.pt')
    common = ['--rank', '1', '--dataset', 'tiny', '--path', str(tmp_path), '--metric', 'ndcg@5', '--test_neg_n', '100',
              '--gpu', '0', '--optimizer', 'Adam', '--lr', '0.001']
    main = os.path.join(ROOT, 'src', 'main.py')
    r = subprocess.run([sys.executable, main, '--model_name', 'IPSBiasedMF', '--epoch', '2', '--model_path', ckpt,
                        '--log_file', str(tmp_path / 'mf.log'), '--result_file', str(tmp_path / 'mf.npy')] + common,
                       capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    log = open(str(tmp_path / 'mf.log')).read()
    assert 'Epoch     2' in log and 'ndcg@5' in log
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'export_exposure.py'), '--path', str(tmp_path),
                        '--dataset', 'tiny', '--model_path', ckpt, '--block_users', '300'],
                       capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    dense = np.load(str(tmp_path / 'tiny' / 'tiny.ips_expo_prob.npy'))
    f = dict(np.load(str(tmp_path / 'tiny' / 'tiny.ipsmf.npz')))
    assert dense.shape == (U, I) and dense.dtype == np.float32
    want = ((f['mf_user'].astype(np.float64) @ f['mf_item'].T.astype(np.float64) + f['mf_user_bias'][:, None]
             + f['mf_item_bias'][None, :] + float(f['mf_global_bias'])) / np.maximum(f['propensity'], f['mf_min_propensity']))
    assert rel_err(dense, want) < 1e-5
    r = subprocess.run([sys.executable, main, '--model_name', 'DCCF', '--epoch', '1', '--model_path',
                        str(tmp_path / 'dccf.pt'), '--log_file', str(tmp_path / 'dccf.log'), '--result_file',
                        str(tmp_path / 'dccf.npy')] + common, capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    assert 'Epoch     1' in open(str(tmp_path / 'dccf.log')).read()
    # DCCF fed the factor file == DCCF fed the dense file (noise-free scoring, same confounders)
    from dccf_b200.models.DCCF import DCCF
    feat = np.load(str(tmp_path / 'tiny' / ('tiny_%s.npy' % synth.DEFAULT_SENTENCE_MODEL)))
    preds = []
    for kw in ({'expo_factors': f}, {'expo_prob': dense}):
        torch.manual_seed(3)
        m = DCCF(path='', dataset='', sentence_model='', sample_num=10, attribute_num=2, std=0.0, label_min=0,
                 label_max=1, feature_num=0, user_num=U, item_num=I, u_vector_size=64, i_vector_size=64, n_layers=1,
                 random_seed=3, model_path='/tmp/unused.pt', feature_embedding=feat, **kw)
        m.apply(m.init_paras)
        m = m.cuda()
        rs = np.random.RandomState(8)
        X = np.stack([rs.randint(0, U, 512), rs.randint(0, I, 512)], 1).astype(np.int64)
        si = torch.from_numpy(rs.randint(0, I, (512, 10)).astype(np.int64))
        preds.append(m.predict({'X': torch.from_numpy(X).cuda(), 'rank': 1, 'train': False, 'dropout': 0.0,
                                'sample_item': si})['prediction'].cpu().numpy())
    assert rel_err(preds[0], preds[1]) < 3e-5
