"""Without a GPU: the launch geometry the float64 reference test of the training step (test_gpu_train_step_reference.py)
relies on, pinned to the library's own host functions, and negative controls of its elementwise comparator — a float32
rounding of the reference passes, and each of the subtle defects a kernel of the step could have is rejected."""
import ctypes

import numpy as np
import pytest

from dccf_b200 import _lib, build
from test_gpu_train_step_reference import (C, CASES, D, UNIT, Case, bounds, bwd_geometry, compare, cross_check_with_oracle,
                                           fwd_ksplits_for, make_problem, mid_smem_bytes, n_rows_of, reference,
                                           simt_geometry, split_rows)


@pytest.fixture(scope='module')
def lib():
    build.build()
    return _lib.load()


def test_geometry_mirror_equals_the_library(lib):
    lib.dccf_train_fused_smem_bytes.restype = ctypes.c_int64
    for F in (64, 128, 192, 384, 768, 960, 1024, 2048):
        for n in list(range(0, 400, 7)) + [1888, 1890, 1920, 2304, 2305, 3280, 3712, 3713, 6272, 6273, 9472, 9473,
                                           11264, 100000]:
            assert lib.dccf_train_fwd_ksplits(n, F) == fwd_ksplits_for(n, F), (n, F)
            if n > 0:
                assert lib.dccf_train_bwd_splits(n, F) == bwd_geometry(n, F)[1], (n, F)
            assert lib.dccf_bwd_splits(n) == simt_geometry(n)[0], n
    for S in list(range(0, 200, 3)) + [118, 119, 120, 180, 181]:
        for A in (1, 2, 3):
            for loss in (0, 1):
                assert lib.dccf_train_fused_smem_bytes(S, A, loss) == mid_smem_bytes(S, A, loss), (S, A, loss)


def test_every_case_reaches_the_geometry_it_claims(lib):
    lib.dccf_train_fused_smem_bytes.restype = ctypes.c_int64
    for c in CASES:
        N = n_rows_of(c)
        assert lib.dccf_train_fwd_ksplits(N, c.F) == fwd_ksplits_for(N, c.F) == c.ks, c.name
        assert lib.dccf_train_bwd_splits(N, c.F) == bwd_geometry(N, c.F)[1] == c.splits, c.name
        assert (lib.dccf_train_fused_smem_bytes(c.S, c.A, c.loss) <= 200 * 1024) == c.fused, c.name
        assert ('fused' in c.paths) == c.fused, c.name
        assert c.fused or 'tc' in c.paths, c.name            # past the limit: the unfused pair is what runs
    case = {c.name: c for c in CASES}
    # the K splits 1, 2, 3, 5, 8 and ks = the number of K chunks (F=64: 4)
    assert {1, 2, 3, 5, 8} <= {c.ks for c in CASES}
    assert any(c.F == 64 and c.ks == 4 for c in CASES)
    # feature widths; 192 and 960 leave a last M tile of the dW kernel that holds only the bias column
    assert {64, 192, 384, 768, 960, 1024, 2048} <= {c.F for c in CASES}
    for F in (192, 960):
        assert (D + F) % 128 == 0 and bwd_geometry(1000, F)[0] == (D + F) // 128 + 1
    # middle kernel: multi-pass phase A (npc * R > 48 rows), multi-pass C1 / C2 (npc * Z > 48), > 48 KB, the limits
    assert any(2 * (c.S + 1) * c.A > 48 and c.fused and c.loss == 0 for c in CASES)
    c40 = case['ks5_s40a2']
    assert 2 * (c40.S + 1) > 48 and mid_smem_bytes(c40.S, c40.A, 0) > 48 * 1024
    assert mid_smem_bytes(119, 2, 0) == 203616 and case['ks8_s119a2'].fused
    assert mid_smem_bytes(120, 2, 0) > 200 * 1024 and not case['s120a2_unfused'].fused
    assert mid_smem_bytes(180, 1, 0) == 204656 and case['s180a1'].fused and not case['s181a1_unfused'].fused
    assert {(c.S, c.A) for c in CASES} >= {(0, 1), (10, 2), (10, 3), (40, 2), (119, 2), (120, 2), (180, 1), (181, 1)}
    # the dW kernel's 60 row splits of 32 rows, the last of 2
    c60 = case['splits60_last2']
    mt, ns, rps = bwd_geometry(n_rows_of(c60), c60.F)
    lo, hi = split_rows(n_rows_of(c60), ns, rps)[-1]
    assert (ns, rps, hi - lo) == (60, 32, 2)
    # losses, random-stream modes, exposure, user shard
    assert any(c.loss == 0 and c.P == 2 for c in CASES) and any(c.loss == 0 and c.P >= 512 for c in CASES)
    assert {c.P for c in CASES if c.loss == 1} >= {1, 3} and any(c.loss == 1 and c.mse_pairs > c.P for c in CASES)
    assert {(c.noise, c.mask) for c in CASES} == {(n, m) for n in range(3) for m in range(3)}
    assert {'dense', 'ipsmf', 'wide'} <= {c.expo for c in CASES}
    assert any(c.user_base != 0 for c in CASES)
    assert {'fused', 'tc', 'simt'} == {p for c in CASES for p in c.paths}


def test_the_bound_has_teeth():
    """C * 2^-20 stays at or below 2^-16 (16 ulps of float32 per unit of the absolute-value computation)."""
    assert 0 < C * UNIT <= 2.0 ** -16


# ------------------------------------------------------------------------------------------------------------------
# negative controls: the comparator on a float32 rounding of the reference, with and without a defect
# ------------------------------------------------------------------------------------------------------------------
CTL = Case('control', 128, 24, 3, 2, 0, 1, 1, 'ipsmf', 5, 0, False, (), 0, 0, True)


@pytest.fixture(scope='module')
def control():
    pb = make_problem(CTL, seed=3)
    N = n_rows_of(CTL)
    _, ns, rps = bwd_geometry(N, CTL.F)
    splits = split_rows(N, ns, rps)
    assert len(splits) >= 2
    return pb, splits


def _as_kernel_output(ref):
    out = {k: np.asarray(ref[k]).astype(np.float32) for k in ('pred', 'dpre', 'gu', 'gi', 'gW', 'gb')}
    out['save_h'] = ref['h'].astype(np.float32)
    out['save_w'] = ref['w'].astype(np.float32)
    out['loss'] = float(np.float32(ref['loss']))
    out['ku'], out['ki'] = ref['ku'].copy(), ref['ki'].copy()
    return out


def _judge(pb, splits, out, noise=None):
    ref = reference(pb, pb['noise'] if noise is None else noise, pb['mask'], CTL.P, splits, save_h=out['save_h'])
    return compare(out, ref)[0]


def test_comparator_accepts_a_float32_rounding_of_the_reference(control):
    pb, splits = control
    ref = reference(pb, pb['noise'], pb['mask'], CTL.P, splits)
    cross_check_with_oracle(ref, pb, pb['mask'])
    assert _judge(pb, splits, _as_kernel_output(ref)) == []


def _defect(pb, splits, name):
    """A float32 rounding of the reference with one defect."""
    noise, mask, K = pb['noise'], pb['mask'], D + CTL.F
    if name == 'last K chunk dropped':
        W = pb['W'].copy()
        W[:, K - 32:] = 0
        return _as_kernel_output(reference(pb, noise, mask, CTL.P, splits, W=W))
    if name == 'noise shifted by one row':
        return _as_kernel_output(reference(pb, np.roll(noise, 1, axis=0), mask, CTL.P, splits))
    if name == 'bias of one column missing':
        b = pb['b'].copy()
        b[37] = 0
        return _as_kernel_output(reference(pb, noise, mask, CTL.P, splits, b=b))
    ref = reference(pb, noise, mask, CTL.P, splits)
    out = _as_kernel_output(ref)
    if name == 'row at a split boundary in the neighbouring partial':
        r = splits[1][0]
        moved = np.outer(ref['dpre'][r], ref['x'][r])
        out['gW'][0] = (ref['gW'][0] + moved).astype(np.float32)
        out['gW'][1] = (ref['gW'][1] - moved).astype(np.float32)
    elif name == 'gate flipped far from the kink':
        pre, bound = ref['pre'], C * UNIT * ref['absP']
        r, c = np.argwhere((pre < -100 * bound) & (ref['m'] != 0))[0]
        out['dpre'][r, c] = np.float32(ref['ds_r'][r] * ref['eu_r'][r, c] * ref['m'][r, c])
    elif name in ('item record scaled by 1 + 1e-4', 'user record scaled by 1 + 1e-4'):
        # the record whose largest element is largest next to its bound
        k = 'gi' if name.startswith('item') else 'gu'
        rec = int(np.argmax((np.abs(ref[k]) / (bounds(ref, C * UNIT)[k] + 1e-300)).max(axis=1)))
        out[k][rec] = (ref[k][rec] * (1 + 1e-4)).astype(np.float32)
    else:
        raise KeyError(name)
    return out


DEFECTS = ['last K chunk dropped', 'noise shifted by one row', 'row at a split boundary in the neighbouring partial',
           'bias of one column missing', 'gate flipped far from the kink', 'item record scaled by 1 + 1e-4',
           'user record scaled by 1 + 1e-4']


@pytest.mark.parametrize('defect', DEFECTS)
def test_comparator_rejects_a_subtle_defect(control, defect):
    pb, splits = control
    assert _judge(pb, splits, _defect(pb, splits, defect)), defect
