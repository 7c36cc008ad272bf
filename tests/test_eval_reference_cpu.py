"""Without a GPU: the launch geometry the float64 reference test of the evaluation kernels (test_gpu_eval_reference.py)
relies on, pinned to the library's host functions where one exists, the routes its cases claim, and negative controls
of its comparators — a float32 rounding of the reference passes, and each of the subtle defects an evaluation kernel
could have is rejected."""
import numpy as np
import pytest

from dccf_b200 import _lib, build
from test_gpu_eval_reference import (C, D, DUP, FS_BN, FS_CASES, SCORER_CASES, UNIT, SCase, abs_bounds,
                                     allowed_items, check_topk, dup_targets, fs_bound, fs_geometry, fs_inputs,
                                     fs_kernel, fs_reference, fwd_bounds, gather_chunks, make_fs_problem,
                                     make_scorer_problem, n_rows, operand_index, scorer_reference, simt_kernel, tf32_hi,
                                     topk_of)
from test_gpu_train_step_reference import compare


@pytest.fixture(scope='module')
def lib():
    build.build()
    return _lib.load()


def test_full_scores_geometry_mirror_equals_the_library(lib):
    for U in (1, 2, 127, 128, 129, 255, 256, 300, 1000, 5000, 18944, 40000, 100000):
        for I in (1, 31, 32, 33, 63, 64, 65, 127, 640, 1000, 4097, 9472, 38048):
            splits, tps, tiles, empty = fs_geometry(U, I)
            assert lib.dccf_full_scores_splits(U, I) == 2 * splits, (U, I)
            # the tiles the splits cover: every tile exactly once, the empty splits at the end
            covered = [t for s in range(splits) for t in range(s * tps, min((s + 1) * tps, tiles))]
            assert covered == list(range(tiles)), (U, I)
            assert empty == sum(1 for s in range(splits) if s * tps >= tiles), (U, I)
    assert lib.dccf_full_scores_ws_floats(4097) == 65 * (2 * (2 * FS_BN * 32 + FS_BN * 8))


def test_every_case_reaches_the_route_it_claims():
    # the SIMT switch: 37 760 rows is the last of k_row_scores_splitk, 37 761 the first of k_row_scores
    assert simt_kernel(37760) == 'k_row_scores_splitk' and simt_kernel(37761) == 'k_row_scores'
    for c in SCORER_CASES:
        N = n_rows(c)
        if c.scorer == 'simt':
            assert c.kernel == '%s<%d>' % (simt_kernel(N), c.noise), c.name
        elif c.scorer.startswith('tc'):
            assert c.kernel == 'k_row_scores_tc<%d>' % c.noise and c.noise in (1, 2), c.name
        else:
            assert c.kernel == 'k_gather_scores' and c.noise == 0 and c.mask == 0, c.name
        for z in c.max_slots:
            assert z <= c.S, c.name
    simt = [c for c in SCORER_CASES if c.scorer == 'simt']
    tc = [c for c in SCORER_CASES if c.scorer == 'tc']
    gather = [c for c in SCORER_CASES if c.scorer == 'gather']
    # SIMT: both sides of the switch at R = 1 and R = 22; rows % 32; every noise x mask mode
    for R in (1, 22):
        sides = {simt_kernel(n_rows(c)) for c in simt if (c.S + 1) * c.A == R}
        assert sides == {'k_row_scores_splitk', 'k_row_scores'}, R
        assert any(abs(n_rows(c) - 37760) <= R and n_rows(c) > 37760 for c in simt if (c.S + 1) * c.A == R)
    assert {n_rows(c) % 32 for c in simt} >= {1, 31}
    assert {(c.noise, c.mask) for c in simt} == {(n, m) for n in range(3) for m in range(3)}
    # tensor cores: rows % 128, F, noise 1 / 2 x mask 0 / 1 / 2, R = 1, the projected operand
    assert {n_rows(c) % 128 for c in tc} >= {0, 1, 127}
    assert {c.F for c in tc} >= {64, 128, 768, 1024}
    assert {(c.noise, c.mask) for c in tc} == {(n, m) for n in (1, 2) for m in range(3)}
    assert any((c.S + 1) * c.A == 1 for c in tc)
    assert any(c.scorer == 'tc_projected' for c in SCORER_CASES)
    # gather: Z, its chunks, n_pairs, the maximum in chunk 2 / 3, wide exposure, IPS-MF, a user shard
    assert {c.S + 1 for c in gather} >= {1, 16, 17, 32, 33, 41}
    assert {gather_chunks(c.S + 1) for c in gather} >= {1, 2, 3}
    assert {c.P for c in gather} >= {1, 15, 16, 17} and any(c.P % 2 == 1 and c.P > 17 for c in gather)
    assert {z // 16 for c in gather for z in c.max_slots} >= {0, 1, 2}
    assert {c.expo for c in gather} >= {'wide', 'ipsmf', 'dense'} and any(c.user_base for c in gather)
    # the backdoor sum: R, A = 3, dense / IPS-MF / wide exposure
    assert {(c.S + 1) * c.A for c in SCORER_CASES} >= {1, 31, 32, 33, 64, 82}
    assert any(c.A == 3 for c in SCORER_CASES) and any(c.S == 40 and c.A == 2 for c in SCORER_CASES)
    assert {c.expo for c in simt} >= {'dense', 'ipsmf', 'wide'}
    # full catalogue: shapes, empty splits, KCAP 8 / 16, k > n_items, ragged last tiles, exclusion
    assert {c.I for c in FS_CASES} >= {1, 31, 32, 33, 64, 65, 4097}
    assert {c.U for c in FS_CASES} >= {1, 127, 128, 129}
    assert any(fs_geometry(c.U, c.I)[3] == 3 for c in FS_CASES if (c.U, c.I) == (5000, 640))
    assert {c.k for c in FS_CASES} >= {1, 8, 9, 16}
    assert {fs_kernel(c.k, c.excl) for c in FS_CASES} >= {fs_kernel(k, e) for k in (0, 8, 9) for e in (False, True)
                                                          if k or not e}
    assert any(c.k > c.I for c in FS_CASES)
    assert {c.I % 64 for c in FS_CASES} >= {1, 31, 32, 33, 0}
    assert {c.kind for c in FS_CASES} == {'ipsmf', 'dccf'}
    # duplicated items in the other column half and in another split
    c = [c for c in FS_CASES if c.I == 4097][0]
    splits, tps, _, _ = fs_geometry(c.U, c.I)
    halves = {(t % 64) // 32 for t in dup_targets(c.I)}
    assert halves == {0, 1} and len({t // 64 // tps for t in dup_targets(c.I)}) >= 3


def test_operand_layout_covers_the_image():
    """operand_index maps W_f's D x F elements onto the hi halves of the chunk images, each float exactly once."""
    for F in (64, 768, 1024):
        idx = operand_index(F).reshape(-1)
        hi = np.concatenate([np.arange(c * 4096, c * 4096 + 2048) for c in range(F // 32)])
        assert np.array_equal(np.sort(idx), hi)


def test_the_bound_has_teeth():
    """C * 2^-20 stays at or below 2^-16 (16 ulps of float32 per unit of the absolute-value computation)."""
    for scorer, outs in C.items():
        for k, c in outs.items():
            assert 0 < c * UNIT <= 2.0 ** -16, (scorer, k)


# ------------------------------------------------------------------------------------------------------------------
# negative controls: the comparators on a float32 rounding of the reference, with and without a defect
# ------------------------------------------------------------------------------------------------------------------
TC_CTL = SCase('tc_control', 'tc', 64, 6, 20, 2, 1, 1, 'wide', 0, (18, 3, 20), 'k_row_scores_tc<1>')
SIMT_CTL = SCase('simt_control', 'simt', 128, 5, 4, 2, 1, 1, 'ipsmf', 0, (), 'k_row_scores_splitk<1>')
GATHER_CTL = SCase('gather_control', 'gather', 64, 7, 36, 2, 0, 0, 'wide', 0, (20, 35, 17), 'k_gather_scores')


def _problem(c):
    return make_scorer_problem(c)


def _judge(c, pb, got, noise=None, mask=None):
    ref, absv = scorer_reference(c, pb, pb.get('noise') if noise is None else noise,
                                 pb.get('mask') if mask is None else mask)
    cc = C['tc' if c.scorer.startswith('tc') else c.scorer]
    got = {k: v for k, v in got.items() if k in cc}          # the outputs this scorer has
    fails, _ = compare(got, ref, c=cc, bounds_fn=fwd_bounds, outputs=('pred', 'save_h', 'save_w'))
    if absv:
        fails += compare(got, ref, c=cc, bounds_fn=abs_bounds(absv), outputs=tuple(absv))[0]
    return fails


def _as_kernel_output(ref):
    out = {'pred': ref['pred'].astype(np.float32), 'save_h': ref['h'].astype(np.float32),
           'save_w': ref['w'].astype(np.float32)}
    if 'dbg_pre' in ref:
        out['dbg_pre'] = ref['dbg_pre'].astype(np.float32)
    return out


def _from_pre(ref, pre):
    """The forward after the pre-activations, in float64: ReLU, dropout, the dot with E_user, the backdoor sum."""
    P, Z, A = ref['P'], ref['Z'], ref['A']
    h = np.maximum(pre, 0) * ref['m']
    s = (h * ref['eu_r']).sum(axis=1).reshape(P, Z, A)
    return h, (ref['w'][:, :, None] * s).sum(axis=1).mean(axis=1)


def _with_noise_product(c, pb, product):
    """A kernel output whose W_f·eps accumulator is `product` (float64 [N, D]) instead of the exact one."""
    ref, _ = scorer_reference(c, pb, pb['noise'], pb['mask'])
    h, pred = _from_pre(ref, ref['pre'] - ref['dbg_pre'] + product)
    out = _as_kernel_output(ref)
    out.update({'pred': pred.astype(np.float32), 'save_h': h.astype(np.float32), 'dbg_pre': product.astype(np.float32)})
    return out


def _split(x):
    hi = tf32_hi(x).astype(np.float64)
    return hi, np.asarray(x, np.float64) - hi


def _scorer_defect(name):
    if name in ('1xTF32 noise product', '2xTF32 noise product (lo x hi dropped)', 'PF without b',
                'noise from row r + 1', 'backdoor sum missing 1/A'):
        c = TC_CTL
    elif name == 'gather softmax with earlier chunks not rescaled':
        c = GATHER_CTL
    else:
        c = SIMT_CTL
    pb = _problem(c)
    noise, mask = pb.get('noise'), pb.get('mask')
    ref, _ = scorer_reference(c, pb, noise, mask)
    out = _as_kernel_output(ref)
    if name.endswith('noise product') or name.endswith('dropped)'):
        nh, nl = _split(noise)
        wh, wl = _split(pb['W'][:, D:])
        prod = nh @ wh.T
        if name.startswith('2x'):
            prod = prod + nh @ wl.T
        return c, pb, _with_noise_product(c, pb, prod)
    if name == 'PF without b':
        h, pred = _from_pre(ref, ref['pre'] - pb['b'].astype(np.float64))
        out.update({'pred': pred.astype(np.float32)})
    elif name == 'noise from row r + 1':
        bad, _ = scorer_reference(c, pb, np.roll(noise, -1, axis=0), mask)
        out = _as_kernel_output(bad)
    elif name == 'backdoor sum missing 1/A':
        out['pred'] = (ref['pred'] * c.A).astype(np.float32)
    elif name == 'dropout quad of the wrong column pair':
        perm = np.arange(D).reshape(-1, 4)[:, [2, 3, 0, 1]].reshape(-1)
        bad, _ = scorer_reference(c, pb, noise, mask[:, perm])
        out = _as_kernel_output(bad)
    elif name == 'gather softmax with earlier chunks not rescaled':
        # every chunk's exponentials are taken against the running maximum of that chunk and never rescaled
        v = O_exposure(pb, ref)
        P, Z = v.shape
        s = ref['s'].mean(axis=2)
        num, den = np.zeros(P), np.zeros(P)
        run = np.full(P, -np.inf)
        for z0 in range(0, Z, 16):
            run = np.maximum(run, v[:, z0:z0 + 16].max(axis=1))
            e = np.exp(v[:, z0:z0 + 16] - run[:, None])
            num += (e * s[:, z0:z0 + 16]).sum(axis=1)
            den += e.sum(axis=1)
        out['pred'] = (num / den).astype(np.float32)
    else:
        raise KeyError(name)
    return c, pb, out


def O_exposure(pb, ref):
    from oracle import dccf_oracle as O
    return O.exposure_values(pb['expo'].astype(np.float64), ref['u'], ref['items'])


SCORER_DEFECTS = ['1xTF32 noise product', '2xTF32 noise product (lo x hi dropped)', 'PF without b',
                  'noise from row r + 1', 'dropout quad of the wrong column pair',
                  'gather softmax with earlier chunks not rescaled', 'backdoor sum missing 1/A']


@pytest.mark.parametrize('c', [TC_CTL, SIMT_CTL, GATHER_CTL], ids=lambda c: c.name)
def test_comparator_accepts_a_float32_rounding_of_the_reference(c):
    pb = _problem(c)
    ref, _ = scorer_reference(c, pb, pb.get('noise'), pb.get('mask'))
    if c.max_slots:
        assert np.array_equal(np.argmax(ref['w'], axis=1), [c.max_slots[p % 3] for p in range(c.P)])
    out = _as_kernel_output(ref)
    if c.scorer == 'tc':
        # the kernel's own arithmetic: 3xTF32 noise product (lo x lo dropped), float32 rounding of what follows
        nh, nl = _split(pb['noise'])
        wh, wl = _split(pb['W'][:, D:])
        out = _with_noise_product(c, pb, nh @ wh.T + nh @ wl.T + nl @ wh.T)
    assert _judge(c, pb, out) == []


@pytest.mark.parametrize('defect', SCORER_DEFECTS)
def test_comparator_rejects_a_subtle_scorer_defect(defect):
    c, pb, out = _scorer_defect(defect)
    assert _judge(c, pb, out), defect


# the full catalogue: one small IPS-MF problem with duplicated items in both column halves and two splits
FS_CTL = FS_CASES[[c.name for c in FS_CASES].index('u128_i65_k9')]._replace(kind='ipsmf', name='fs_control')


def _fs_control():
    return make_fs_problem(FS_CTL)[0]


def _fs_emulated(p, drop=None):
    """The kernel's product on the augmented operands A' = [A, fl(rb + g), 1], B' = [fl(cs B), cs, fl(cs cb)], split
    into TF32 hi / lo parts: hi·hi + hi·lo + lo·hi (drop: 'lo' = the correction terms, 'lohi' = one of them)."""
    A, Bs, rbg, cs, cbs = fs_inputs(p)
    Aa = np.concatenate([A, rbg[:, None], np.ones((A.shape[0], 1), np.float32)], axis=1)
    Ba = np.concatenate([Bs, cs[:, None], cbs[:, None]], axis=1)
    ah, al = _split(Aa)
    bh, bl = _split(Ba)
    M = ah @ bh.T
    if drop != 'lo':
        M = M + ah @ bl.T
        if drop != 'lohi':
            M = M + al @ bh.T
    return M.astype(np.float32)


def _fs_judge(p, M, ts=None, ti=None, k=9):
    ref, absv = fs_reference(p)
    fails = compare({'scores': M}, {'scores': ref}, c=C['fs'], bounds_fn=abs_bounds({'scores': absv}),
                    outputs=('scores',))[0]
    if ti is not None:
        fails += check_topk(ts, ti, M, ref, fs_bound(ref, absv), k, allowed_items(M.shape[1], M.shape[0], None))
    return fails


def test_full_scores_comparator_accepts_the_kernel_arithmetic():
    p = _fs_control()
    # copies of items 0..7 in the other column half of tile 0 and in split 1
    splits, tps, _, _ = fs_geometry(FS_CTL.U, FS_CTL.I)
    assert splits == 2 and {(i // 64 // tps, (i % 64) // 32) for t in [0] + dup_targets(FS_CTL.I)
                            for i in range(t, t + DUP)} >= {(0, 0), (0, 1), (1, 0)}
    for M in (fs_reference(p)[0].astype(np.float32), _fs_emulated(p)):
        ts, ti = topk_of(M, 9, allowed_items(M.shape[1], M.shape[0], None))
        # the lists hold exact ties (duplicated items), broken by ascending id
        assert any(len(set(ts[u].tolist())) < 9 for u in range(M.shape[0]))
        assert _fs_judge(p, M, ts, ti) == []


FS_DEFECTS = ['1xTF32 product', '2xTF32 product (lo x hi dropped)', 'row_bias added after the column scale',
              'top-k ties ordered by descending id', 'a merge that drops one column half\'s list']


@pytest.mark.parametrize('defect', FS_DEFECTS)
def test_full_scores_comparator_rejects_a_subtle_defect(defect):
    p = _fs_control()
    M = fs_reference(p)[0].astype(np.float32)
    allowed = allowed_items(M.shape[1], M.shape[0], None)
    ts, ti = topk_of(M, 9, allowed)
    if defect == '1xTF32 product':
        M = _fs_emulated(p, drop='lo')
        ts, ti = topk_of(M, 9, allowed)
    elif defect.startswith('2xTF32'):
        M = _fs_emulated(p, drop='lohi')
        ts, ti = topk_of(M, 9, allowed)
    elif defect.startswith('row_bias'):
        M = fs_reference(p, row_bias_after_scale=True)[0].astype(np.float32)
        ts, ti = topk_of(M, 9, allowed)
    elif defect.startswith('top-k ties'):
        ts, ti = topk_of(M, 9, allowed, desc_ties=True)
        assert not np.array_equal(ti, topk_of(M, 9, allowed)[1])
    else:
        half0 = [a[(a % 64) < 32] for a in allowed]
        ts, ti = topk_of(M, 9, half0)
    assert _fs_judge(p, M, ts, ti), defect
