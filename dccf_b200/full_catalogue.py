"""Full-catalogue scoring on the tcgen05 tensor cores (dccf_full_scores) — the one dense user x item GEMM of
the path (BASELINE.json config 4; SURVEY.md §8a row 16) — and evaluation over the whole catalogue.

* `ipsmf_exposure(factors)` — the IPSBiasedMF prediction of every (user, item) pair
  (src/models/IPSBiasedMF.py:37-57): `(<p_u,q_i> + b_u + b_i + g) / max(propensity_i, M)`.  README.md:27-29 of the
  reference: this matrix is what DCCF loads as `<dataset>.ips_expo_prob.npy`.
* `ipsmf_topk(factors, k, exclude)` — the same scores, per-user top-k only (the matrix is never written).
* `dccf_catalogue_topk(model, k, users, exclude)` — deterministic DCCF scores of the whole catalogue (std 0, no
  confounder items): `score[u,i] = <E_user[u], relu(W_i·E_item[i] + W_f·Feat[i] + b)>`.
* `known_items_csr(user_his, users, n_items)` — per-user item lists as the CSR the kernels read.
* `evaluate_full_catalogue(model_or_factors, data_loader, metrics, split)` — ndcg / hit / precision / recall / f1 @k
  of the held-out items against every item the user has not interacted with, one GPU or user-sharded under torchrun.
"""
import numpy as np
import torch

from . import kernels

METRIC_COLUMN = {'ndcg': 0, 'hit': 1, 'precision': 2, 'recall': 3, 'f1': 4}


def _col_scale(factors):
    prop = factors['propensity']
    return 1.0 / torch.clamp(prop, min=float(factors['mf_min_propensity']))


def _device_csr(csr, dev):
    off, items = csr
    return (torch.as_tensor(off, dtype=torch.int64).to(dev).contiguous(),
            torch.as_tensor(items, dtype=torch.int32).to(dev).contiguous())


def ipsmf_exposure(factors):
    """[U,I] float32 exposure matrix from IPSBiasedMF factors (dict of CUDA tensors, keys as in
    dccf_b200.synth.make_ipsmf_factors)."""
    out, _, _ = kernels.full_scores(factors['mf_user'], factors['mf_item'], factors['mf_user_bias'],
                                    factors['mf_item_bias'], _col_scale(factors), float(factors['mf_global_bias']),
                                    materialise=True, k=0)
    return out


def ipsmf_topk(factors, k, exclude=None):
    """Per-user top-k of the IPSBiasedMF scores.  exclude = (off [U+1], items) CSR over the rows of factors['mf_user']
    (known_items_csr): those items never enter the row's list."""
    ex = None if exclude is None else _device_csr(exclude, factors['mf_user'].device)
    _, s, i = kernels.full_scores(factors['mf_user'], factors['mf_item'], factors['mf_user_bias'],
                                  factors['mf_item_bias'], _col_scale(factors), float(factors['mf_global_bias']),
                                  materialise=False, k=k, exclude=ex)
    return s, i


def dccf_catalogue_topk(model, k, users=None, exclude=None):
    """Top-k items per user over the WHOLE catalogue with the deterministic DCCF predictor.  users: rows of the user
    table (None: all); exclude = (off, items) CSR over those rows (known_items_csr)."""
    if model.sample_num != 0 or model.std != 0:
        raise ValueError('full-catalogue DCCF scoring is a GEMM only without confounder samples and feature noise '
                         '(sample_num == 0, std == 0); got sample_num=%d std=%g' % (model.sample_num, model.std))
    model._check_ready()
    t = model._tc_tables()
    hidden = torch.relu(t['PI'] + t['PF']).contiguous()
    A = model.uid_embeddings.weight.data if users is None else model.uid_embeddings.weight.data[users].contiguous()
    ex = None if exclude is None else _device_csr(exclude, A.device)
    _, s, i = kernels.full_scores(A, hidden, materialise=False, k=k, exclude=ex)
    return s, i


def _csr_from_pairs(rows, items, n_rows, n_items):
    """Sorted, de-duplicated CSR (int64 offsets, int32 items) of (row, item) pairs."""
    key = np.sort(rows.astype(np.int64) * n_items + items.astype(np.int64))
    key = key[np.concatenate(([True], key[1:] != key[:-1]))] if key.size else key
    off = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(key // n_items, minlength=n_rows), out=off[1:])
    return off, (key % n_items).astype(np.int32)


def known_items_csr(user_his, users, n_items):
    """CSR of the items of `users` (in that order) in `user_his` — a {uid: [iid, ...]} dict such as
    DataLoader.train_user_his, or a sequence of such dicts whose lists are united.  Returns (off int64 [len(users)+1],
    items int32): each row sorted ascending and de-duplicated.  An id outside [0, n_items) raises."""
    his = [user_his] if isinstance(user_his, dict) else list(user_his)
    users = np.asarray(users, dtype=np.int64)
    order = np.argsort(users, kind='stable')
    rows, items = [np.zeros(0, dtype=np.int64)], [np.zeros(0, dtype=np.int64)]
    for h in his:
        keys = np.fromiter(h.keys(), dtype=np.int64, count=len(h))
        lens = np.fromiter((len(v) for v in h.values()), dtype=np.int64, count=len(h))
        flat = np.concatenate([np.asarray(v, dtype=np.int64) for v in h.values()] + [np.zeros(0, dtype=np.int64)])
        at = np.minimum(np.searchsorted(users[order], keys), max(len(users) - 1, 0))
        hit = (users[order][at] == keys) if len(users) else np.zeros(len(keys), dtype=bool)
        take = np.repeat(hit, lens)
        rows.append(np.repeat(order[at] if len(users) else at, lens)[take])
        items.append(flat[take])
    rows, items = np.concatenate(rows), np.concatenate(items)
    if items.size and (items.min() < 0 or items.max() >= n_items):
        raise ValueError('item id outside [0, %d) in a user history' % n_items)
    return _csr_from_pairs(rows, items, len(users), n_items)


def _rows_of(off):
    return np.repeat(np.arange(len(off) - 1, dtype=np.int64), np.diff(off))


def _minus(a, b, n_items):
    """Row-wise set difference a \\ b of two CSRs over the same rows."""
    ka = _rows_of(a[0]) * n_items + a[1]
    kb = _rows_of(b[0]) * n_items + b[1]
    keep = ~np.isin(ka, kb, assume_unique=True)
    return _csr_from_pairs(_rows_of(a[0])[keep], a[1][keep], len(a[0]) - 1, n_items)


def _take_rows(csr, rows):
    off, items = csr
    cnt = np.diff(off)[rows]
    new_off = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum(cnt, out=new_off[1:])
    idx = np.repeat(off[rows] - new_off[:-1], cnt) + np.arange(new_off[-1], dtype=np.int64)
    return new_off, items[idx]


def _split_his(df, label):
    """{uid: item array} of the rows of an interaction frame with a positive label."""
    if label in df.columns:
        df = df[df[label] > 0]
    uid, iid = df['uid'].to_numpy(np.int64), df['iid'].to_numpy(np.int64)
    order = np.argsort(uid, kind='stable')
    users, starts = np.unique(uid[order], return_index=True)
    return {int(u): it for u, it in zip(users.tolist(), np.split(iid[order], starts[1:]))}


def _parse_metrics(metrics):
    out = []
    for m in metrics:
        name, _, k = m.partition('@')
        if name not in METRIC_COLUMN or not k.isdigit() or not 1 <= int(k) <= kernels.RANK_STREAM_MAX_K:
            raise ValueError('full-catalogue evaluation computes <name>@k with name in %s and 1 <= k <= %d; got %r'
                             % ('/'.join(METRIC_COLUMN), kernels.RANK_STREAM_MAX_K, m))
        out.append((METRIC_COLUMN[name], int(k)))
    return out


def evaluation_sets(data_loader, split, n_items):
    """(users, exclude CSR, positives CSR) of a full-catalogue evaluation, users ascending.  Excluded: the user's
    training items, plus the validation items for split='test'.  Positives: the split's items minus the excluded ones;
    users without a positive are left out."""
    if split not in ('test', 'validation'):
        raise ValueError("split must be 'test' or 'validation', got %r" % (split,))
    label = data_loader.label
    split_his = _split_his(data_loader.test_df if split == 'test' else data_loader.validation_df, label)
    users = np.array(sorted(split_his), dtype=np.int64)
    excl_src = [data_loader.train_user_his]
    if split == 'test':
        excl_src.append(_split_his(data_loader.validation_df, label))
    excl = known_items_csr(excl_src, users, n_items)
    pos = _minus(known_items_csr(split_his, users, n_items), excl, n_items)
    keep = np.nonzero(np.diff(pos[0]) > 0)[0]
    return users[keep], _take_rows(excl, keep), _take_rows(pos, keep)


def evaluate_full_catalogue(model_or_factors, data_loader, metrics, split='test'):
    """Ranking metrics over the whole catalogue, in the order of `metrics`, averaged over the evaluated users (as
    BaseModel.evaluate_method averages over users).  metrics: '<name>@k', name in ndcg / hit / precision / recall / f1,
    k <= 16.

    Every item the user interacted with in training (and, for split='test', in validation) is removed before ranking.
    The positives are the user's items of the split minus those: a held-out item the user also has in training cannot
    be ranked, so it is not a positive.  Users without a positive are not evaluated.

    model_or_factors: IPSBiasedMF factors (dict of CUDA tensors, dccf_b200.synth.make_ipsmf_factors keys) or a DCCF
    model scored with the deterministic predictor (sample_num == 0, std == 0; see dccf_catalogue_topk).  A checkpoint
    trained with confounders and feature noise evaluates this way: build the model with sample_num=0, std=0 (the
    state-dict keys do not depend on them) and load_model() the checkpoint.

    Under torchrun every rank scores a contiguous block of the evaluated users; the metric sums and the user count are
    all-reduced (dccf_b200.dist.all_reduce_sum)."""
    from .dist import all_reduce_sum, is_distributed
    want = _parse_metrics(metrics)
    ks = sorted(set(k for _, k in want))
    factors = model_or_factors if isinstance(model_or_factors, dict) else None
    if factors is not None:
        dev, n_items = factors['mf_user'].device, factors['mf_item'].shape[0]
    else:
        model = model_or_factors
        if model.user_shard is not None:
            raise NotImplementedError('full-catalogue evaluation needs the whole user table on every rank')
        dev, n_items = model.uid_embeddings.weight.device, model.item_num
    users, excl, pos = evaluation_sets(data_loader, split, n_items)
    rank, world = (torch.distributed.get_rank(), torch.distributed.get_world_size()) if is_distributed() else (0, 1)
    lo, hi = len(users) * rank // world, len(users) * (rank + 1) // world
    sums = np.zeros((len(ks), 5), dtype=np.float64)
    count = 0
    if hi > lo:
        block = np.arange(lo, hi)
        u = torch.from_numpy(users[lo:hi]).to(dev)
        ex = _take_rows(excl, block)
        if factors is not None:
            sub = dict(factors, mf_user=factors['mf_user'][u].contiguous(),
                       mf_user_bias=factors['mf_user_bias'][u].contiguous())
            _, ids = ipsmf_topk(sub, ks[-1], exclude=ex)
        else:
            _, ids = dccf_catalogue_topk(model, ks[-1], users=u, exclude=ex)
        po, pi = _device_csr(_take_rows(pos, block), dev)
        out = torch.empty((len(ks), 5), dtype=torch.float64, device=dev)
        n = torch.empty(1, dtype=torch.int64, device=dev)
        for a in range(0, len(ks), kernels.RANK_MAX_NK):
            group = ks[a:a + kernels.RANK_MAX_NK]
            kernels.topk_metrics(ids, po, pi, group, out_sums=out[a:a + len(group)], out_count=n)
        sums, count = out.cpu().numpy(), int(n.item())
    tot = all_reduce_sum(list(sums.ravel()) + [count])
    n_users = max(1.0, float(tot[-1]))
    return [float(tot[ks.index(k) * 5 + col] / n_users) for col, k in want]
