"""Full-catalogue evaluation on the GPU: the fused top-k with known-item exclusion, dccf_topk_metrics, and
evaluate_full_catalogue end to end (one GPU, a checkpoint trained with confounders, two ranks)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from dccf_b200 import full_catalogue as fc
from dccf_b200 import kernels, synth
from oracle import dccf_oracle as O
from test_full_catalogue_cpu import metric_case

pytestmark = pytest.mark.gpu

METRICS = ['ndcg@5', 'hit@5', 'precision@5', 'recall@10', 'f1@10', 'ndcg@16']


def _ipsmf(U, I, dup=True, seed=4):
    f = synth.make_ipsmf_factors(U, I, seed=seed)
    if dup:      # items 100..199 repeat items 0..99 exactly: exact score ties, broken by item id
        for key in ('mf_item', 'mf_item_bias', 'propensity'):
            f[key][100:200] = f[key][0:100]
    return {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else float(v)) for k, v in f.items()}


def _excl_lists(U, I, k, seed=1):
    rs = np.random.RandomState(seed)
    lists = []
    for u in range(U):
        n = [0, 3, 40, 300][u % 4]
        lists.append(sorted(rs.choice(I, size=n, replace=False).tolist()))
    lists[7] = sorted(set(range(I)) - {5, 105, I - 1})            # three rankable items: padded with -1
    lists[8] = list(range(64, 128)) + list(range(I - 20, I))      # whole tile, partial last tile
    off = np.zeros(U + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(l) for l in lists])
    return lists, (off, np.array([i for l in lists for i in l], dtype=np.int32))


def _np_topk(M, lists, k):
    """float64 top-k of the device's own scores over the non-excluded items (score desc, item id asc)."""
    U, I = M.shape
    ids = -np.ones((U, k), dtype=np.int64)
    sc = np.full((U, k), -np.inf, dtype=np.float32)
    for u in range(U):
        cand = np.setdiff1d(np.arange(I), np.asarray(lists[u], dtype=np.int64))
        s = M[u, cand].astype(np.float64)
        top = cand[np.lexsort((cand, -s))[:k]]
        ids[u, :len(top)] = top
        sc[u, :len(top)] = M[u, top]
    return sc, ids


def _dccf(U, I, S=0, std=0.0, path='', dataset='', seed=2019, model_path='/tmp/unused.pt'):
    from dccf_b200.models.DCCF import DCCF
    rs = np.random.RandomState(seed)
    feat = (rs.standard_normal((I, 768)) / np.sqrt(768)).astype(np.float32) if not path else None
    expo = rs.random_sample((U, I)).astype(np.float32) if not path else None
    torch.manual_seed(seed)
    m = DCCF(path=path, dataset=dataset, sentence_model=synth.DEFAULT_SENTENCE_MODEL, sample_num=S, attribute_num=2,
             std=std, label_min=0, label_max=1, feature_num=0, user_num=U, item_num=I, u_vector_size=64,
             i_vector_size=64, n_layers=1, random_seed=seed, model_path=model_path, feature_embedding=feat,
             expo_prob=expo)
    m.apply(m.init_paras)
    return m.cuda()


def _dccf_matrix(model, users=None):
    t = model._tc_tables()
    hidden = torch.relu(t['PI'] + t['PF']).contiguous()
    A = model.uid_embeddings.weight.data
    A = A if users is None else A[users].contiguous()
    return kernels.full_scores(A, hidden, materialise=True, k=0)[0].cpu().numpy()


@pytest.mark.parametrize('k', [1, 5, 8, 16])
@pytest.mark.parametrize('scorer', ['ipsmf', 'dccf'])
def test_topk_with_exclusion_equals_numpy(k, scorer):
    torch.cuda.set_device(0)
    U, I = 300, 1000                                    # neither a multiple of the 128 x 64 tile
    lists, csr = _excl_lists(U, I, k)
    if scorer == 'ipsmf':
        f = _ipsmf(U, I)
        M = fc.ipsmf_exposure(f).cpu().numpy()
        p = f['mf_user'].double() @ f['mf_item'].double().T + f['mf_user_bias'].double()[:, None] \
            + f['mf_item_bias'].double()[None, :] + f['mf_global_bias']
        p = (p / torch.clamp(f['propensity'].double(), min=f['mf_min_propensity'])[None, :]).cpu().numpy()
        assert np.abs(M - p).max() / np.abs(p).max() < 1e-5
        s, i = fc.ipsmf_topk(f, k, exclude=csr)
    else:
        model = _dccf(400, I)
        with torch.no_grad():                           # exact ties: duplicated item rows
            model.iid_embeddings.weight[100:200] = model.iid_embeddings.weight[0:100]
            model.feature_embedding[100:200] = model.feature_embedding[0:100]
        users = torch.arange(399, 399 - U, -1, device='cuda')        # a subset of the table, in reverse order
        M = _dccf_matrix(model, users)
        s, i = fc.dccf_catalogue_topk(model, k, users=users, exclude=csr)
    want_s, want_i = _np_topk(M, lists, k)
    got_i = i.cpu().numpy()
    assert np.array_equal(got_i, want_i)
    assert np.array_equal(s.cpu().numpy(), want_s)
    assert (got_i[7] == -1).sum() == max(0, k - 3) and set(got_i[7][got_i[7] >= 0]) <= {5, 105, I - 1}
    for u in range(U):
        assert not set(got_i[u].tolist()) & set(lists[u])


@pytest.mark.parametrize('k', [5, 16])
def test_no_exclusion_is_unchanged(k):
    torch.cuda.set_device(0)
    f = _ipsmf(300, 1000)
    base = fc.ipsmf_topk(f, k)
    none = fc.ipsmf_topk(f, k, exclude=None)
    empty = fc.ipsmf_topk(f, k, exclude=(np.zeros(301, dtype=np.int64), np.zeros(0, dtype=np.int32)))
    for a in (none, empty):
        for x, y in zip(base, a):
            assert torch.equal(x, y)
    with pytest.raises(kernels._lib.DccfError, match='fused top-k only'):
        ex = fc._device_csr((np.zeros(301, dtype=np.int64), np.zeros(1, dtype=np.int32)), 'cuda')
        kernels.full_scores(f['mf_user'], f['mf_item'], materialise=True, k=k, exclude=ex)


def test_topk_metrics_equal_the_oracle():
    torch.cuda.set_device(0)
    ks = [1, 5, 10, 16]
    topk, pos_sets, (scores, uid, labels, iids) = metric_case(seed=11, n_users=300)
    counted = [g for g in range(len(topk)) if pos_sets[g]]
    off = np.zeros(len(topk) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(p) for p in pos_sets])
    items = np.array([i for p in pos_sets for i in sorted(p)], dtype=np.int32)
    po, pi = fc._device_csr((off, items), 'cuda')
    ids = torch.from_numpy(topk).cuda()
    per = torch.empty((len(topk), len(ks), 5), dtype=torch.float64, device='cuda')
    sums = torch.empty((len(ks), 5), dtype=torch.float64, device='cuda')
    n = torch.empty(1, dtype=torch.int64, device='cuda')
    kernels.topk_metrics(ids, po, pi, ks, out_metrics=per, out_sums=sums, out_count=n)
    per, sums = per.cpu().numpy(), sums.cpu().numpy()
    assert int(n.item()) == len(counted)
    assert np.isnan(per[[g for g in range(len(topk)) if not pos_sets[g]]]).all()
    for j, k in enumerate(ks):
        users, _, _, want = O.rank_users(scores, uid, labels, iids, k)
        assert users.tolist() == counted
        np.testing.assert_allclose(per[counted, j], want, rtol=0, atol=1e-12)
        np.testing.assert_allclose(sums[j], want.sum(axis=0), rtol=1e-12, atol=1e-12)


def _reference_eval(M, dl, metrics, split):
    """The numpy evaluation from a materialised [U,I] score matrix: every non-excluded item is a candidate."""
    users, (eo, ei), (po, pi) = fc.evaluation_sets(dl, split, M.shape[1])
    scores, uid, labels, iids = [], [], [], []
    for r, u in enumerate(users.tolist()):
        cand = np.setdiff1d(np.arange(M.shape[1]), ei[eo[r]:eo[r + 1]])
        scores.append(M[u, cand]); uid.append(np.full(len(cand), u)); iids.append(cand)
        labels.append(np.isin(cand, pi[po[r]:po[r + 1]]).astype(np.float32))
    scores, uid, labels, iids = (np.concatenate(x) for x in (scores, uid, labels, iids))
    return O.evaluate_method(scores, {'uid': uid, 'Y': labels, 'iid': iids}, metrics)


def _toy(tmp_path, U=300, I=700, seed=3):
    from dccf_b200.data_loaders.DataLoader import DataLoader
    root = str(tmp_path / 'datasets')
    synth.write_dataset(root, 'toy', n_users=U, n_items=I, per_user=12, feat_dim=768, seed=seed)
    return root, DataLoader(path=root, dataset='toy', label='label', sep=',')


@pytest.mark.parametrize('split', ['test', 'validation'])
def test_evaluate_full_catalogue_equals_numpy(tmp_path, split):
    torch.cuda.set_device(0)
    _, dl = _toy(tmp_path)
    f = _ipsmf(dl.user_num, dl.item_num, dup=False)
    got = fc.evaluate_full_catalogue(f, dl, METRICS, split=split)
    want = _reference_eval(fc.ipsmf_exposure(f).cpu().numpy(), dl, METRICS, split)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    with pytest.raises(ValueError):
        fc.evaluate_full_catalogue(f, dl, ['ndcg@17'])
    with pytest.raises(ValueError):
        fc.evaluate_full_catalogue(f, dl, ['auc'])


def test_checkpoint_trained_with_confounders_evaluates_deterministically(tmp_path):
    torch.cuda.set_device(0)
    root, dl = _toy(tmp_path, U=200, I=500)
    ckpt = str(tmp_path / 'm.pt')
    d = os.path.join(root, 'toy')
    trained = _dccf(dl.user_num, dl.item_num, S=10, std=0.1, path=d, dataset='toy', model_path=ckpt)
    trained.optimizer = trained.make_fused_optimizer(lr=1e-2, l2=1e-4)
    rs = np.random.RandomState(0)
    X = np.stack([rs.randint(0, dl.user_num, 64), rs.randint(0, dl.item_num, 64)], 1).astype(np.int64)
    trained.train_step({'X': torch.from_numpy(X).cuda(), 'Y': torch.cat([torch.ones(32), torch.zeros(32)]).cuda(),
                        'rank': 1, 'train': True, 'dropout': 0.0})
    trained.save_model()
    with pytest.raises(ValueError, match='sample_num == 0'):
        fc.evaluate_full_catalogue(trained, dl, METRICS)
    model = _dccf(dl.user_num, dl.item_num, S=0, std=0.0, path=d, dataset='toy', seed=7, model_path=ckpt)
    model.load_model()
    for key, v in trained.state_dict().items():
        assert torch.equal(model.state_dict()[key], v), key
    got = fc.evaluate_full_catalogue(model, dl, METRICS)
    want = _reference_eval(_dccf_matrix(model), dl, METRICS, 'test')
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    # the command-line entry point on the same checkpoint
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'full_catalogue_eval.py'), '--path', root + '/',
                        '--dataset', 'toy', '--sep', ',', '--model_path', ckpt, '--metric', ','.join(METRICS)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    np.testing.assert_allclose([line['metrics'][m] for m in METRICS], got, rtol=1e-12, atol=1e-12)


def test_two_rank_sharded_evaluation_equals_one_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    torch.cuda.set_device(0)
    root, dl = _toy(tmp_path, U=301, I=700)
    ckpt = str(tmp_path / 'm.pt')
    model = _dccf(dl.user_num, dl.item_num, path=os.path.join(root, 'toy'), dataset='toy', model_path=ckpt)
    model.save_model()
    one = fc.evaluate_full_catalogue(model, dl, METRICS)
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', '29531', os.path.join(ROOT, 'tools', 'full_catalogue_eval.py'), '--path',
           root + '/', '--dataset', 'toy', '--sep', ',', '--model_path', ckpt, '--metric', ','.join(METRICS)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line['n_gpus'] == 2
    np.testing.assert_allclose([line['metrics'][m] for m in METRICS], one, rtol=1e-12, atol=1e-12)
