"""Full-catalogue evaluation without a GPU: the exclusion / positive sets, a lock-step emulation of the fused top-k's
exclusion cursor, the top-k metric definitions against the oracle, and the ctypes argument lists of the two entry
points against include/dccf_b200.h."""
import ctypes
import os
import re
import types

import numpy as np
import pandas as pd
import pytest

from conftest import ROOT
from dccf_b200 import _lib, full_catalogue as fc, synth
from oracle import dccf_oracle as O


@pytest.fixture(scope='module')
def tiny_loader(tmp_path_factory):
    from dccf_b200.data_loaders.DataLoader import DataLoader
    root = str(tmp_path_factory.mktemp('datasets'))
    synth.write_dataset(root, 'toy', n_users=60, n_items=300, per_user=12, feat_dim=8, seed=5)
    return DataLoader(path=root, dataset='toy', label='label', sep=',')


def _rows(df, u):
    return set(df.loc[(df['uid'] == u) & (df['label'] > 0), 'iid'].tolist())


@pytest.mark.parametrize('split', ['test', 'validation'])
def test_known_items_and_positives_on_a_synth_dataset(tiny_loader, split):
    dl = tiny_loader
    users, (eo, ei), (po, pi) = fc.evaluation_sets(dl, split, dl.item_num)
    assert eo.dtype == np.int64 and po.dtype == np.int64 and ei.dtype == np.int32 and pi.dtype == np.int32
    assert np.all(np.diff(users) > 0) and len(eo) == len(po) == len(users) + 1
    held = dl.test_df if split == 'test' else dl.validation_df
    for r, u in enumerate(users.tolist()):
        ex, pos = ei[eo[r]:eo[r + 1]], pi[po[r]:po[r + 1]]
        assert np.all(np.diff(ex) > 0) and np.all(np.diff(pos) > 0)          # sorted and unique
        want_ex = set(dl.train_user_his.get(u, [])) | (_rows(dl.validation_df, u) if split == 'test' else set())
        assert set(ex.tolist()) == want_ex
        assert set(pos.tolist()) == _rows(held, u) - want_ex and len(pos) > 0
    assert set(users.tolist()) == {u for u in held['uid'].unique().tolist() if _rows(held, u)}
    # the same CSR straight from the public helper, for an explicit user order with duplicates in the histories
    off, items = fc.known_items_csr([{1: [5, 3, 5]}, {1: [3, 9], 7: [2]}], [7, 4, 1], 10)
    assert off.tolist() == [0, 1, 1, 4] and items.tolist() == [2, 3, 5, 9]
    with pytest.raises(ValueError):
        fc.known_items_csr({0: [10]}, [0], 10)


def test_positives_lose_excluded_items_and_empty_users_are_dropped():
    frame = lambda rows: pd.DataFrame(rows, columns=['uid', 'iid', 'label', 'time'])
    dl = types.SimpleNamespace(
        label='label', train_user_his={0: [1, 2], 1: [4], 2: [7]},
        train_df=None,
        validation_df=frame([(0, 3, 1, 0), (1, 5, 1, 0), (2, 8, 0, 0)]),
        test_df=frame([(0, 2, 1, 0), (0, 6, 1, 0), (1, 4, 1, 0), (1, 5, 1, 0), (2, 9, 1, 0), (3, 1, 0, 0)]))
    users, (eo, ei), (po, pi) = fc.evaluation_sets(dl, 'test', 10)
    # user 0: 2 is a training item -> positive {6}; user 1: 4 in train, 5 in validation -> dropped;
    # user 2: the zero-label validation row is no interaction; user 3: no positive label at all
    assert users.tolist() == [0, 2]
    assert [ei[eo[r]:eo[r + 1]].tolist() for r in range(2)] == [[1, 2, 3], [7]]
    assert [pi[po[r]:po[r + 1]].tolist() for r in range(2)] == [[6], [9]]
    users, (eo, ei), (po, pi) = fc.evaluation_sets(dl, 'validation', 10)
    assert users.tolist() == [0, 1] and pi.tolist() == [3, 5] and ei.tolist() == [1, 2, 4]
    with pytest.raises(ValueError):
        fc.evaluation_sets(dl, 'train', 10)


# ---- lock-step emulation of the exclusion cursor of k_full_scores<TOPK, KCAP, true> -------------------------------
FS_BM, FS_BN = 128, 64


def _splits(n_users, n_items):                      # dccf_full_scores_splits / 2
    ut, it = -(-n_users // FS_BM), -(-n_items // FS_BN)
    return max(1, min((2 * 148 + ut - 1) // ut, it))


def _emulate_thread(lst, c, c_end, t_lo, t_hi, chalf):
    """One epilogue thread: binary search once, then per tile the merge loop; returns the excluded items it masked
    and asserts every read is inside [c, c_end)."""
    first = t_lo * FS_BN
    lo, hi = c, c_end
    while lo < hi:
        mid = (lo + hi) >> 1
        assert c <= mid < c_end
        if lst[mid] < first:
            lo = mid + 1
        else:
            hi = mid
    c = lo
    INF = 2 ** 31 - 1
    nxt = lst[c] if c < c_end else INF
    masked = []
    for t in range(t_lo, t_hi):
        i0 = t * FS_BN + chalf * 32
        mask = 0
        while nxt < i0 + 32:
            if nxt >= i0:
                mask |= 1 << (nxt - i0)
            c += 1
            assert c <= c_end
            nxt = lst[c] if c < c_end else INF
        masked += [i0 + j for j in range(32) if mask >> j & 1]
    return masked


def _emulate(off, items, n_items):
    n_users = len(off) - 1
    splits = _splits(n_users, n_items)
    n_tiles = -(-n_items // FS_BN)
    tps = -(-n_tiles // splits)
    got = [[] for _ in range(n_users)]
    for s in range(splits):
        t_lo, t_hi = s * tps, min(s * tps + tps, n_tiles)
        for u in range(n_users):
            for chalf in (0, 1):
                got[u] += _emulate_thread(items, int(off[u]), int(off[u + 1]), t_lo, t_hi, chalf)
    return got


@pytest.mark.parametrize('n_users,n_items', [(300, 1000), (40, 38000 // 16), (129, 64 * 7), (2000, 38000 // 16)])
def test_exclusion_cursor_masks_exactly_the_listed_items(n_users, n_items):
    rs = np.random.RandomState(n_users)
    splits = _splits(n_users, n_items)
    n_tiles = -(-n_items // FS_BN)
    tps = -(-n_tiles // splits)
    assert splits > 1
    lists = []
    for u in range(n_users):
        kind = u % 5
        if kind == 0:
            lst = []                                                          # empty list
        elif kind == 1:                                                       # whole tiles (and a whole split)
            t = rs.randint(n_tiles)
            lst = list(range(t * FS_BN, min((t + 2) * FS_BN, n_items)))
        elif kind == 2:                                                       # across a split boundary
            b = min(tps, n_tiles - 1) * FS_BN
            lst = list(range(max(0, b - 40), min(n_items, b + 40)))
        elif kind == 3:                                                       # the partial last tile
            lst = list(range(max(0, n_items - 37), n_items))
        else:
            lst = sorted(rs.choice(n_items, size=rs.randint(1, 60), replace=False).tolist())
        lists.append(lst)
    off = np.zeros(n_users + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(l) for l in lists])
    items = np.array([i for l in lists for i in l], dtype=np.int64)
    got = _emulate(off, items, n_items)
    for u in range(n_users):
        assert sorted(got[u]) == lists[u], u                                  # each item masked exactly once


def test_exclusion_cursor_stays_in_bounds_on_an_unsorted_list():
    rs = np.random.RandomState(3)
    n_items = 1000
    lists = [rs.randint(0, n_items, size=50).tolist() for _ in range(20)]
    off = np.zeros(21, dtype=np.int64)
    off[1:] = np.cumsum([len(l) for l in lists])
    items = np.array([i for l in lists for i in l], dtype=np.int64)
    got = _emulate(off, items, n_items)                                        # asserts every read in range
    for u in range(20):
        assert set(got[u]) <= set(lists[u])


# ---- the top-k metric definitions --------------------------------------------------------------------------------
def topk_metrics_reference(topk_id, pos_sets, ks):
    """[n_users, len(ks), 5] with NaN for users without a positive: the definitions dccf_topk_metrics applies."""
    out = np.full((len(topk_id), len(ks), 5), np.nan)
    for g, (ids, pos) in enumerate(zip(topk_id, pos_sets)):
        if not pos:
            continue
        n_pos = len(pos)
        for j, k in enumerate(ks):
            rel = np.array([1.0 if (i >= 0 and i in pos) else 0.0 for i in ids[:k]])
            disc = 1.0 / np.log2(np.arange(2, k + 2))
            hits = rel.sum()
            out[g, j] = [(rel * disc).sum() / disc[:min(n_pos, k)].sum(), float(hits > 0), hits / k, hits / n_pos,
                         2 * hits / (k + n_pos)]
    return out


def metric_case(seed=11, n_users=40, n_items=120):
    """Ranked lists of length 16 over a catalogue with per-user exclusions (some -1 padded, many score ties), each
    user's positives (some users without one), and the explicit candidate lists of the users with a positive
    (scores, uid, labels, iids) as oracle.rank_users takes them."""
    rs = np.random.RandomState(seed)
    topk, pos_sets, scores, uid, labels, iids = [], [], [], [], [], []
    for g in range(n_users):
        excl = set(rs.choice(n_items, size=rs.randint(0, 30), replace=False).tolist())
        if g % 7 == 3:                                   # fewer than 16 rankable items: the list is -1 padded
            excl = set(range(n_items)) - set(range(g % 5, g % 5 + 9))
        rank_ok = np.array(sorted(set(range(n_items)) - excl))
        s = rs.randint(0, 6, size=len(rank_ok)).astype(np.float32)          # many exact ties
        pos = set(rs.choice(rank_ok, size=min(len(rank_ok), rs.randint(0 if g % 9 == 0 else 1, 8)),
                            replace=False).tolist())
        order = np.lexsort((rank_ok, -s.astype(np.float64)))
        ids = -np.ones(16, dtype=np.int64)
        ids[:min(16, len(order))] = rank_ok[order[:16]]
        topk.append(ids)
        pos_sets.append(pos)
        if pos:
            scores.append(s); uid.append(np.full(len(s), g)); iids.append(rank_ok)
            labels.append(np.array([1.0 if i in pos else 0.0 for i in rank_ok], dtype=np.float32))
    return np.array(topk), pos_sets, tuple(np.concatenate(x) for x in (scores, uid, labels, iids))


def test_topk_metric_definitions_equal_the_oracle_on_the_full_candidate_list():
    ks = [1, 5, 10, 16]
    topk, pos_sets, (scores, uid, labels, iids) = metric_case()
    got = topk_metrics_reference(topk, pos_sets, ks)
    counted = [g for g in range(len(topk)) if pos_sets[g]]
    assert np.isnan(got[[g for g in range(len(topk)) if not pos_sets[g]]]).all()
    for j, k in enumerate(ks):
        users, want_ids, _, want = O.rank_users(scores, uid, labels, iids, k)
        assert users.tolist() == counted
        assert np.array_equal(want_ids, topk[counted][:, :k])
        np.testing.assert_allclose(got[counted, j], want, rtol=0, atol=1e-12)


# ---- ctypes argument lists of the entry points against the header --------------------------------------------------
_CTYPE = {'int32_t': ctypes.c_int32, 'int64_t': ctypes.c_int64, 'int': ctypes.c_int, 'float': ctypes.c_float,
          'double': ctypes.c_double, 'uint64_t': ctypes.c_uint64}


@pytest.mark.parametrize('name', ['dccf_full_scores', 'dccf_topk_metrics', 'dccf_rank_eval_multi'])
def test_ctypes_argument_lists_match_the_header(name):
    header = re.sub(r'/\*.*?\*/', '', open(os.path.join(ROOT, 'include', 'dccf_b200.h')).read(), flags=re.S)
    m = re.search(r'\b(\w+)\s+' + name + r'\s*\(([^)]*)\)\s*;', header)
    assert m, name
    params = [p.strip() for p in m.group(2).split(',')]
    res, args = _lib._SIGNATURES[name]
    assert res is _CTYPE[m.group(1)]
    assert len(args) == len(params), (name, len(args), len(params))
    for p, a in zip(params, args):
        if '*' in p:
            base = p.replace('const', '').split('*')[0].strip()
            assert a is _lib._P or (base in _CTYPE and a is ctypes.POINTER(_CTYPE[base])), (name, p, a)
        else:
            assert a is _CTYPE[p.split()[0]], (name, p, a)


def test_entry_points_reject_bad_arguments_before_any_cuda_call():
    from dccf_b200 import build
    build.build()
    lib = _lib.load()
    p = 4096                                            # never dereferenced: argument checks come first
    rc = lib.dccf_full_scores(8, 8, p, p, None, None, None, 0.0, p, 5, p, p, p, p, p, p, p, None)
    assert rc == -1 and b'fused top-k only' in lib.dccf_last_error()
    rc = lib.dccf_full_scores(8, 8, p, p, None, None, None, 0.0, None, 5, p, p, p, p, p, p, None, None)
    assert rc == -1 and b'both excl_off and excl_items' in lib.dccf_last_error()
    ks = (ctypes.c_int32 * 2)(5, 10)
    rc = lib.dccf_topk_metrics(p, 4, 8, p, p, ks, 2, None, p, p, None, None)
    assert rc == -1 and b'k=10 outside [1,8]' in lib.dccf_last_error()
    rc = lib.dccf_topk_metrics(p, 4, 17, p, p, ks, 2, None, p, p, None, None)
    assert rc == -1 and b'list length 17' in lib.dccf_last_error()
