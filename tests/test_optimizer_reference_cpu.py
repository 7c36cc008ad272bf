"""Without a GPU: the launch geometry the float64 reference test of the optimizer step (test_gpu_optimizer_reference.py)
relies on, pinned to the library's own CTA assignment (dccf_adam_blocks), the geometry each of its cases claims, and
negative controls of its elementwise comparator — a float32 rounding of the reference passes, and each of the defects an
optimizer kernel could have is rejected."""
import ctypes

import numpy as np
import pytest

from dccf_b200 import _lib, build
from test_gpu_optimizer_reference import (ALL, C, CASES, D, LIST_CAP, UNIT, WIDTHS, Case, blocks, compare, dense_sums,
                                          make_problem, records_of, reference, row_sums, sweep_warps)


@pytest.fixture(scope='module')
def lib():
    build.build()
    return _lib.load()


def lib_blocks(lib, mode, rows, recs, dense_n):
    nt, nd = len(rows), len(dense_n)
    arr = lambda t, xs: (t * max(1, len(xs)))(*xs)      # noqa: E731
    lo, bn = (ctypes.c_int32 * max(1, nt + nd))(), (ctypes.c_int32 * max(1, nt + nd))()
    grid = lib.dccf_adam_blocks(mode, arr(ctypes.c_int64, rows), arr(ctypes.c_int64, recs), nt, arr(ctypes.c_int64, dense_n),
                                nd, lo, bn)
    return [(lo[i], bn[i]) for i in range(nt + nd)], grid


def test_geometry_mirror_equals_the_library(lib):
    rs = np.random.RandomState(0)
    configs = [([1568, 30000], [1024, 11264], [64 * 832, 64]), ([1], [0], [1]), ([0], [0], []), ([], [], [257]),
               ([3, 1202, 1], [64, 384, 0], [257, 255]), ([10 ** 7, 10 ** 6], [65536, 720896], [64 * 2112, 64])]
    for _ in range(300):
        nt, nd = rs.randint(0, 5), rs.randint(0, 5)
        configs.append((list(rs.randint(0, 10 ** rs.randint(1, 8), nt)), list(rs.randint(0, 10 ** rs.randint(1, 6), nt)),
                        list(rs.randint(0, 10 ** rs.randint(1, 7), nd))))
    for rows, recs, dense_n in configs:
        for mode in range(4):
            assert lib_blocks(lib, mode, rows, recs, dense_n) == blocks(mode, rows, recs, dense_n), (mode, rows, recs, dense_n)
    assert lib.dccf_adam_blocks(4, None, None, 0, None, 0, None, None) == -1
    assert lib.dccf_adam_blocks(0, None, None, 5, None, 0, None, None) == -1
    for rows, recs, dense_n in (([-1], [0], []), ([4], [-1], []), ([4], [0], [-1])):
        assert lib_blocks(lib, 2, rows, recs, dense_n)[1] == -1
    # only mode 2 reads the record counts
    for mode in (0, 1, 3):
        assert lib_blocks(lib, mode, [100, 5000], [7, 70000], [64]) == lib_blocks(lib, mode, [100, 5000], [0, 0], [64])


def _geometry(c):
    """What one case reaches: per-table record counts, touched rows, and the sweeps' CTA ranges."""
    pb = make_problem(c, c.rules[0])
    tabs = pb['tables']
    rows = [t['n_rows'] for t in tabs]
    recs = [len(t['keys']) for t in tabs]
    dense_n = [d['n'] for d in pb['dense']]
    counts = [np.bincount(t['keys'], minlength=t['n_rows']) for t in tabs]
    return pb, rows, recs, dense_n, counts


def test_every_case_reaches_the_geometry_it_claims(lib):
    seen = {k: set() for k in ('rows_mod4', 'counts', 'touched_vs_hw', 'n', 'n_parts', 'n_seg')}
    flags = set()
    for c in CASES:
        pb, rows, recs, dense_n, counts = _geometry(c)
        assert (recs[0], recs[1]) == records_of(c)
        # planted record counts, distinct users, padded segments
        for k in c.i_counts:
            assert k in counts[1], (c.name, k)
        seen['counts'] |= set(c.i_counts)
        if c.u_distinct:
            assert (counts[0] > 0).sum() == c.u_distinct, c.name
            if c.u_distinct == c.U:
                flags.add('every row touched')
        if c.empty:
            assert recs[2] == 0
            flags.add('table without records')
        seen['rows_mod4'] |= {r % 4 for r in rows}
        flags |= {'%d rows' % r for r in rows if r in (1, 3)}
        seen['n_seg'].add((c.n_seg, c.user_seg >= 0, c.pad > 0))
        for n, n_parts, extra in c.dense:
            seen['n'].add(n)
            seen['n_parts'].add(n_parts)
            if extra > 0:
                flags.add('part_stride > n')
        if c.F:
            assert c.dense[0][0] == D * (D + c.F) and c.F % 64 == 0
        # the touched-row sweep (mode 2): touched user rows against the half-warp stride of the user range
        geo, _ = lib_blocks(lib, 2, rows, recs, dense_n)
        hw = geo[0][1] * 256 // 16
        touched = int((counts[0] > 0).sum())
        for name, k in (('1', 1), ('hw', hw), ('hw+1', hw + 1), ('2hw', 2 * hw), ('2hw+1', 2 * hw + 1)):
            if touched == k:
                seen['touched_vs_hw'].add(name)
        if geo[1][1] < (recs[1] + 15) // 16:
            flags.add('records above the mode-2 CTA budget')
        # the sweeps (modes 0, 1 at every width, 3): a table of exactly 4 * n_warps * trips rows (trips >= 2), and one more
        for mode, widths in ((0, (256,)), (1, [w for w in WIDTHS if w > 0]), (3, (256,))):
            geo, _ = lib_blocks(lib, mode, rows, recs, dense_n)
            for w in widths:
                for r, (_, bn) in zip(rows, geo):
                    per_trip = 4 * sweep_warps(mode, bn, w)
                    if r >= 2 * per_trip and r % per_trip in (0, 1):
                        flags.add('sweep rows %% (4 n_warps) == %d, mode %d' % (r % per_trip, mode))
        if c.edges:
            flags.add('edges')
            t = pb['tables'][1]
            assert np.isnan(t['grads']).any() and np.isinf(t['grads']).any() and (t['grads'] == pb['hp']['clip']).any()
            assert (np.abs(t['p']).max(axis=1) == 0).any() and (np.abs(t['p']).max(axis=1) < 1e-10).any()
            assert ((t['p'] != 0) & (np.abs(t['p']) < np.finfo(np.float32).tiny)).sum() > 64     # subnormal p
        if c.big_eps:
            flags.add('big eps')
    assert seen['rows_mod4'] == {0, 1, 2, 3}
    assert {1, 2, 3, 4, 5, 95, 96, 97, 700} <= seen['counts'] and LIST_CAP == 96
    assert seen['touched_vs_hw'] == {'1', 'hw', 'hw+1', '2hw', '2hw+1'}
    assert {1, 255, 257, 64 * (64 + 768), 64 * (64 + 2048)} <= seen['n']
    assert {1, 15, 16, 17, 20, 33, 60} <= seen['n_parts']
    assert {(1, False, False), (2, False, True), (8, True, True)} <= seen['n_seg']
    for f in ('every row touched', 'table without records', '1 rows', '3 rows', 'part_stride > n', 'edges', 'big eps',
              'records above the mode-2 CTA budget'):
        assert f in flags, f
    for mode in (0, 1, 3):
        for r in (0, 1):
            assert 'sweep rows %% (4 n_warps) == %d, mode %d' % (r, mode) in flags, (mode, r)


def test_every_hyper_parameter_term_is_visible():
    """lr * l2 and lr * wd move a parameter by many ulps, l2 != wd, and some elements clip only through the l2 term."""
    c = CASES[0]
    pb = make_problem(c, 'gd')
    hp = pb['hp']
    assert hp['l2'] != hp['wd']
    p = pb['tables'][1]['p'].astype(np.float64)
    ulp = np.spacing(np.abs(pb['tables'][1]['p']))
    assert np.median(hp['lr'] * hp['wd'] * np.abs(p) / ulp) > 1000
    gs, _, _ = row_sums(pb['tables'][1])
    g1 = gs + 2 * np.float32(hp['l2']) * p
    assert ((np.abs(gs) < hp['clip']) & (np.abs(g1) > hp['clip'])).sum() > 10
    assert ((np.abs(g1) < hp['clip']) & (np.abs(g1 + hp['wd'] * p) > hp['clip'])).sum() > 10


def test_the_bound_has_teeth():
    """C * 2^-20 stays at or below 2^-16 for every output."""
    assert all(0 < c * UNIT <= 2.0 ** -16 for c in C.values())


# ------------------------------------------------------------------------------------------------------------------
# negative controls: the comparator on a float32 rounding of the reference, with and without a defect
# ------------------------------------------------------------------------------------------------------------------
CTL = Case('control', 37, 403, 40, 5, 1, -1, 0, None, (1, 2, 5, 97), ((257, 17, 3), (64, 17, 0)), 0, True, False, 0, ALL)


def _kernel_like(pb, defect=None):
    """A float32 rounding of the reference for every tensor of the problem, with one defect."""
    hp = pb['hp']
    out = []
    for i, x in enumerate(pb['tables'] + pb['dense']):
        is_table = i < len(pb['tables'])
        if is_table:
            t = x
            if defect == 'a row missing one record':
                counts = np.bincount(t['keys'], minlength=t['n_rows'])
                drop = np.flatnonzero(t['keys'] == np.flatnonzero(counts >= 3)[0])[0]
                t = dict(t, keys=np.delete(t['keys'], drop), grads=np.delete(t['grads'], drop, axis=0))
            gs, A, n = row_sums(t)
        else:
            gs, A = dense_sums(x)
        ref = reference(hp, x['p'], x['st'], gs, A, defect=defect)
        with np.errstate(invalid='ignore', over='ignore'):
            o = {'p': (x['p'].astype(np.float64) + ref['p']).astype(np.float32)}
            for k in x['st']:
                o[k] = ref[k].astype(np.float32)
        if defect == 'untouched rows not updated' and is_table:
            idle = np.bincount(x['keys'], minlength=x['n_rows']) == 0
            o['p'][idle] = x['p'][idle]
            for k in x['st']:
                o[k][idle] = x['st'][k][idle]
        out.append(o)
    return out


def _judge(pb, out):
    hp, fails = pb['hp'], 0
    for i, x in enumerate(pb['tables'] + pb['dense']):
        gs, A = row_sums(x)[:2] if i < len(pb['tables']) else dense_sums(x)
        f, _ = compare(hp['rule'], hp, x['p'], x['st'], gs, A, out[i])
        fails += f['any']
    return fails


@pytest.mark.parametrize('rule', ALL)
def test_comparator_accepts_a_float32_rounding_of_the_reference(rule):
    for big_eps in (False, True):
        pb = make_problem(CTL, rule, seed=4, big_eps=big_eps)
        assert _judge(pb, _kernel_like(pb)) == 0, (rule, big_eps)


DEFECTS = ['no weight decay', 'l2 and wd swapped', 'clip before + 2*l2*p', 'clip after + wd*p', 'a row missing one record',
           'untouched rows not updated', 'NaN clipped to -clip']
ADAM_DEFECTS = ['bias correction at t - 1', 'eps inside the square root']


@pytest.mark.parametrize('rule,defect', [(r, d) for r in ALL for d in DEFECTS] + [('adam', d) for d in ADAM_DEFECTS])
def test_comparator_rejects_a_defect(rule, defect):
    pb = make_problem(CTL, rule, seed=4, big_eps=defect == 'eps inside the square root')
    assert _judge(pb, _kernel_like(pb, defect)) > 0, (rule, defect)
