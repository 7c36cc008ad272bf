"""Every kernel that produces an evaluation number, against a float64 reference, element by element, over its launch
geometry: the projected item tables and the split W_f operand of dccf_tc_prepare, the noise-free gather scorer
(dccf_score_gather), the tensor-core scorer (dccf_score_fwd_tc: k_row_scores_tc + k_backdoor, the exact and the
projected noise operand), the FP32 SIMT scorer (dccf_score_fwd) on both sides of its k_row_scores_splitk /
k_row_scores switch, the full-catalogue GEMM and its fused top-k (dccf_full_scores), DCCF.predict_many over a ragged
evaluation set, and the ranker's two fallbacks (more candidates than the staging buffer, massive ties at the threshold).

The reference is fed the exact float32 inputs the kernels use: the noise / masks the library materialises at the call's
seed and offset, fl(Feat + eps) where the kernel adds the noise in float32, and fl(rb_u + g), fl(cs_i * B_i),
fl(cs_i * cb_i) for the full catalogue.  Bound per element (tests/test_gpu_train_step_reference.py):

    |y_kernel - y_ref| <= C * 2^-20 * |y|_abs + ULPS * |y|

|y|_abs is the computation on absolute values with each stage's input bound carried through it to first order.  C is
per scorer and output, about four times the largest value a B200 needs; `observed` (printed per case, and the largest
per output at the end of the module) is the smallest C each output needed.  The route each case claims — which kernel
and which instantiation it runs — is read from a torch.profiler trace of the call itself."""
import collections

import numpy as np
import pytest

from oracle import dccf_oracle as O
from test_gpu_train_step_reference import (D, ULPS, UNIT, Case, _device_problem, compare, forward_bounds,
                                           forward_reference, make_problem)

pytestmark = pytest.mark.gpu

N_SM = 148
FWD_BM, TC_KC, GATHER_CHUNK = 128, 32, 16
FS_BM, FS_BN = 128, 64
STD, P_DROP = 0.1, 0.2
SEED, OFFSET = 2019, 5

# C per scorer and output: about 4 x the largest ratio observed on a B200 (NVIDIA B200, 1000 W power limit).  The
# predictions' bounds are their pre-activations' bounds carried through (the prediction itself never needed more than
# C = 0.006 beyond its 8 ulps), so pred takes the C of its scorer's pre-activations.
C = {'prep': {'PI': 0.4, 'PF': 0.8},                                # observed 0.097, 0.196
     'gather': {'pred': 0.8},                                       # PI + PF
     'tc': {'pred': 0.8, 'dbg_pre': 0.8},                           # observed 0.005, 0.196
     'simt': {'pred': 0.8, 'save_h': 0.8, 'save_w': 0.15},          # observed 0, 0.193, 0.036
     'fs': {'scores': 3.0}}                                         # observed 0.757


# ------------------------------------------------------------------------------------------------------------------
# the launch geometry, mirrored from score_fwd.cu (the splitk switch), gather_scores.cu (16-slot chunks) and
# full_scores.cu (dccf_full_scores_splits, KCAP); tests/test_eval_reference_cpu.py pins what has a host function
# ------------------------------------------------------------------------------------------------------------------
def simt_kernel(n_rows):
    """The row kernel dccf_score_fwd launches for n_rows rows."""
    return 'k_row_scores_splitk' if -(-n_rows // FWD_BM) < 2 * N_SM else 'k_row_scores'


def gather_chunks(Z):
    return -(-Z // GATHER_CHUNK)


def fs_geometry(U, I):
    """(item splits, tiles per split, item tiles, splits that get no tile) of dccf_full_scores."""
    ut, it = -(-U // FS_BM), -(-I // FS_BN)
    if ut <= 0 or it <= 0:
        return 1, 0, 0, 0
    splits = max(1, min(-(-2 * N_SM // ut), it))
    tps = -(-it // splits)
    return splits, tps, it, splits - (-(-it // tps))


def fs_kernel(k, excl):
    if k == 0:
        return 'k_full_scores<false,1,false>'
    return 'k_full_scores<true,%d,%s>' % (8 if k <= 8 else 16, 'true' if excl else 'false')


def tf32_hi(x):
    """The TF32 'hi' part the tensor-core kernels split an operand into: the top 19 bits."""
    return (np.asarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def operand_index(F):
    """[D, F] -> float index of W_f[n, f] in the hi half of its chunk image (k_prep_wf, tc_layout.cuh core_offset);
    the lo part is 2048 floats further."""
    n, f = np.meshgrid(np.arange(D), np.arange(F), indexing='ij')
    c, kk = f // TC_KC, f % TC_KC
    off = ((n >> 3) * 1024 + (kk >> 2) * 128 + (n & 7) * 16 + (kk & 3) * 4) // 4
    return c * 4096 + off


# ------------------------------------------------------------------------------------------------------------------
# cases; each states the route it is meant to reach (checked without a GPU and again in the profiler trace)
# ------------------------------------------------------------------------------------------------------------------
SCase = collections.namedtuple('SCase', 'name scorer F P S A noise mask expo user_base max_slots kernel')
SCORER_CASES = [
    # gather: Z = 1, 16, 17, 32, 33, 41; n_pairs 1, 15, 16, 17, odd; the exposure maximum in chunk 2 / 3
    SCase('g_z1_p1', 'gather', 64, 1, 0, 1, 0, 0, 'dense', 0, (), 'k_gather_scores'),
    SCase('g_z16_p15', 'gather', 768, 15, 15, 2, 0, 0, 'wide', 0, (15,), 'k_gather_scores'),
    SCase('g_z17_p16', 'gather', 64, 16, 16, 1, 0, 0, 'wide', 0, (16,), 'k_gather_scores'),
    SCase('g_z32_p17', 'gather', 128, 17, 31, 1, 0, 0, 'ipsmf', 0, (20, 31), 'k_gather_scores'),
    SCase('g_z33_p33_shard', 'gather', 64, 33, 32, 2, 0, 0, 'wide', 500, (32, 16, 0), 'k_gather_scores'),
    SCase('g_z41_p257', 'gather', 768, 257, 40, 2, 0, 0, 'wide', 0, (16, 40, 33, 5), 'k_gather_scores'),
    # tensor cores: n_rows % 128 in {0, 1, 127}; F 64 / 128 / 768 / 1024; noise 1, 2 x mask 0, 1, 2
    SCase('tc_f64_n1m0', 'tc', 64, 16, 11, 2, 1, 0, 'dense', 0, (), 'k_row_scores_tc<1>'),        # 384 rows
    SCase('tc_f128_n2m2_r1', 'tc', 128, 129, 0, 1, 2, 2, 'dense', 0, (), 'k_row_scores_tc<2>'),   # 129 rows, R = 1
    SCase('tc_f768_n2m1', 'tc', 768, 67, 6, 3, 2, 1, 'ipsmf', 0, (), 'k_row_scores_tc<2>'),       # 1407 rows
    SCase('tc_f1024_n1m2', 'tc', 1024, 257, 0, 1, 1, 2, 'dense', 300, (), 'k_row_scores_tc<1>'),  # 257 rows
    SCase('tc_f768_n2m0', 'tc', 768, 64, 10, 2, 2, 0, 'wide', 0, (), 'k_row_scores_tc<2>'),       # 1408 rows
    SCase('tc_f64_n1m1', 'tc', 64, 16, 3, 2, 1, 1, 'dense', 0, (), 'k_row_scores_tc<1>'),         # 128 rows
    # the projected operand: M [D, D] in place of W_f, D normals per row
    SCase('tc_projected', 'tc_projected', 768, 40, 10, 2, 2, 2, 'dense', 0, (), 'k_row_scores_tc<2>'),
    # SIMT: both sides of the switch at R = 1 and R = 22; n_rows % 32 in {1, 31}; noise x mask; R 31..82 backdoor
    SCase('simt_37760', 'simt', 64, 37760, 0, 1, 0, 0, 'dense', 0, (), 'k_row_scores_splitk<0>'),
    SCase('simt_37761', 'simt', 64, 37761, 0, 1, 2, 2, 'dense', 0, (), 'k_row_scores<2>'),
    SCase('simt_r22_37752', 'simt', 64, 1716, 10, 2, 1, 1, 'dense', 0, (), 'k_row_scores_splitk<1>'),
    SCase('simt_r22_37774', 'simt', 128, 1717, 10, 2, 1, 2, 'ipsmf', 0, (), 'k_row_scores<1>'),
    SCase('simt_r31', 'simt', 768, 1, 30, 1, 2, 0, 'dense', 0, (), 'k_row_scores_splitk<2>'),
    SCase('simt_r33_a3', 'simt', 192, 1, 10, 3, 0, 2, 'dense', 0, (), 'k_row_scores_splitk<0>'),
    SCase('simt_r32', 'simt', 64, 3, 31, 1, 2, 1, 'wide', 0, (), 'k_row_scores_splitk<2>'),
    SCase('simt_r64', 'simt', 64, 5, 31, 2, 1, 0, 'ipsmf', 0, (), 'k_row_scores_splitk<1>'),
    SCase('simt_r82', 'simt', 128, 7, 40, 2, 0, 1, 'wide', 7, (), 'k_row_scores_splitk<0>'),
]
SCASE = {c.name: c for c in SCORER_CASES}


def n_rows(c):
    return c.P * (c.S + 1) * c.A


def as_train_case(c):
    return Case(c.name, c.F, c.P, c.S, c.A, 1, 1 if c.noise == 1 and c.scorer != 'tc_projected' else 0,
                1 if c.mask == 1 else 0, c.expo, c.user_base, 0, False, (), 0, 0, False)


def exposure_table(pb):
    """float64 [U, I] exposure values of every (local user, item)."""
    if 'ipsmf' in pb:
        e = {k: (np.asarray(v, np.float64) if isinstance(v, np.ndarray) else v) for k, v in pb['ipsmf'].items()}
        U, I = e['mf_user'].shape[0], e['mf_item'].shape[0]
        return O.exposure_values(e, np.arange(U), np.tile(np.arange(I), (U, 1)))
    return pb['expo'].astype(np.float64)


def place_max(pb, slots):
    """Move each pair's highest-exposure item into slot slots[p % len(slots)] (and out of every other slot), so that
    the softmax maximum first appears there."""
    V = exposure_table(pb)
    X, si = pb['X'], pb['si']
    I = V.shape[1]
    for p in range(X.shape[0]):
        u = X[p, 0] - pb['user_base']
        best = int(np.argmax(V[u]))
        items = np.concatenate([[X[p, 1]], si[p]])
        items[items == best] = (best + 1) % I
        items[slots[p % len(slots)]] = best
        X[p, 1], si[p] = items[0], items[1:]


def make_scorer_problem(c):
    pb = make_problem(as_train_case(c), seed=17 + 31 * SCORER_CASES.index(c) if c in SCORER_CASES else 3)
    if c.max_slots:
        place_max(pb, c.max_slots)
    return pb


# ------------------------------------------------------------------------------------------------------------------
# float64 reference and bounds
# ------------------------------------------------------------------------------------------------------------------
def fwd_bounds(ref, eps):
    return forward_bounds(ref, eps)[0]


def abs_bounds(absv):
    """bounds_fn of compare() for outputs whose |y|_abs is given directly."""
    return lambda ref, eps: {k: eps * a + ULPS * np.abs(ref[k]) for k, a in absv.items()}


def projected_problem(pb, M):
    """The projected operand as an ordinary problem: x = [E_item | Feat | g] against W = [W_i | W_f | M]."""
    I = pb['Feat'].shape[0]
    q = dict(pb)
    q['Feat'] = np.concatenate([pb['Feat'], np.zeros((I, D), np.float32)], axis=1)
    q['W'] = np.concatenate([pb['W'], M], axis=1)
    q['F'] = pb['F'] + D
    return q


def scorer_reference(c, pb, noise, mask, M=None):
    """Forward reference of one scorer call; for the tensor-core scorers also dbg_pre (the raw W_f·eps accumulator)."""
    if c.scorer == 'tc_projected':
        N = n_rows(c)
        ref = forward_reference(projected_problem(pb, M), np.concatenate([np.zeros((N, c.F), np.float32), noise], 1),
                                mask, noise_exact=True, c=C['tc']['pred'])
        Wn = M.astype(np.float64)
    else:
        ref = forward_reference(pb, noise, mask, noise_exact=c.scorer == 'tc', c=C['simt']['save_h'])
        Wn = pb['W'][:, D:].astype(np.float64)
    absv = {}
    if c.scorer in ('tc', 'tc_projected'):
        n64 = noise.astype(np.float64)
        ref['dbg_pre'] = n64 @ Wn.T
        absv['dbg_pre'] = np.abs(n64) @ np.abs(Wn).T
    return ref, absv


def check_scorer(c, ref, absv, got, label=''):
    key = 'tc' if c.scorer == 'tc_projected' else c.scorer
    cc = C[key]
    fails, observed = compare(got, ref, c=cc, bounds_fn=fwd_bounds, outputs=('pred', 'save_h', 'save_w'))
    if absv:
        f2, o2 = compare(got, ref, c=cc, bounds_fn=abs_bounds(absv), outputs=tuple(absv))
        fails += f2
        observed.update(o2)
    for k, v in observed.items():
        OBSERVED[key, k] = max(OBSERVED[key, k], v)
    print('%-18s %s observed C: %s' % (c.name, label, ' '.join('%s %.3g' % kv for kv in observed.items())))
    assert not fails, '%s:\n  ' % c.name + '\n  '.join(fails)


OBSERVED = collections.defaultdict(float)


@pytest.fixture(scope='module', autouse=True)
def _report_observed():
    yield
    if OBSERVED:
        print('\nlargest C observed: ' + ', '.join('%s.%s %.3g' % (s, o, v) for (s, o), v in sorted(OBSERVED.items())))


# ------------------------------------------------------------------------------------------------------------------
# running the kernels
# ------------------------------------------------------------------------------------------------------------------
def traced(fn):
    """(fn(), names of the CUDA kernels it launched, spaces removed), from a torch.profiler trace."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name.replace(' ', '') for e in prof.events()}


def launched(names, kernel):
    """kernel (e.g. 'k_backdoor', 'k_row_scores<2>') is among the demangled names of a trace."""
    return any(('::' + kernel + '(') in n for n in names)


def _t(a, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def streams(c, pb, dev, width, seed=SEED, offset=OFFSET, materialised=False):
    """(rng, noise values, mask values, tensors to keep alive).  mode 2: the library's materialisers at the call's
    seed / offset give the values; materialised=True feeds those values as mode 1 instead."""
    import torch
    from dccf_b200 import kernels
    N = n_rows(c)
    keep, noise, mask = {}, None, None
    if c.noise == 1 and c.scorer != 'tc_projected':
        keep['noise'] = _t(pb['noise'], dev)
        noise = pb['noise']
    elif c.noise:
        t = kernels.noise_fill(torch.empty((N, width), dtype=torch.float32, device=dev), STD, seed, offset)
        noise = t.cpu().numpy()
        if materialised or c.noise == 1:
            keep['noise'] = t
    if c.mask == 1:
        keep['mask'] = _t(pb['mask'], dev)
        mask = pb['mask']
    elif c.mask == 2:
        t = kernels.dropout_mask_fill(torch.empty((N, D), dtype=torch.float32, device=dev), P_DROP, seed, offset)
        mask = t.cpu().numpy()
        if materialised:
            keep['mask'] = t
    rng = kernels.make_rng(noise=keep.get('noise'), mask=keep.get('mask'), noise_std=STD, p_drop=P_DROP, seed=seed,
                           offset=offset, generate_noise=c.noise == 2 and 'noise' not in keep,
                           generate_mask=c.mask == 2 and 'mask' not in keep)
    return rng, noise, mask, keep


def nan(dev, *shape):
    import torch
    return torch.full(shape, float('nan'), dtype=torch.float32, device=dev)


def prepare(dt, F, dev):
    """dccf_tc_prepare: (PI, PF, gB)."""
    import torch
    from dccf_b200 import kernels
    I = dt['E_item'].shape[0]
    PI, PF = nan(dev, I, D), nan(dev, I, D)
    gB = nan(dev, kernels.tc_operand_floats(F))
    ws_wt = torch.empty((D + F) * D, dtype=torch.float32, device=dev)
    kernels.tc_prepare(dt['dims'], dt['E_item'], dt['Feat'], dt['W'], dt['b'], ws_wt, PI, PF, gB)
    return PI, PF, gB


def projected_operand(M, dev):
    """The operand image of M as DCCF._projected_operand builds it (dccf_tc_prepare on a stand-in problem, F = D)."""
    import torch
    from dccf_b200 import kernels
    Wfake = np.zeros((D, 2 * D), np.float32)
    Wfake[:, D:] = M
    z = torch.zeros((8, D), dtype=torch.float32, device=dev)
    gB = torch.empty(kernels.tc_operand_floats(D), dtype=torch.float32, device=dev)
    kernels.tc_prepare(kernels.make_dims(8, 8, D, 0, 1), z, z, _t(Wfake, dev), torch.zeros(D, device=dev),
                       torch.empty(2 * D * D, dtype=torch.float32, device=dev), torch.empty_like(z),
                       torch.empty_like(z), gB)
    return gB


def run_scorer(c, dt, rng, dev, tables=None, gBp=None, extra=0):
    """One call of the case's scorer; outputs as numpy (+ 'err' and the buffers' tails past n_pairs)."""
    import torch
    from dccf_b200 import kernels
    P, N, Z, F = c.P, n_rows(c), c.S + 1, c.F
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    pred = nan(dev, P + extra)
    out = {}
    if c.scorer == 'gather':
        PI, PF, _ = tables
        kernels.score_gather(dt['dims'], dt['E_user'], PI, PF, dt['expo'], dt['X'], dt['si'], pred, err)
    elif c.scorer in ('tc', 'tc_projected'):
        PI, PF, gB = tables
        dims = dt['dims']
        if gBp is not None:
            gB = gBp
            dims = kernels.make_dims(dt['E_user'].shape[0], dt['E_item'].shape[0], D, c.S, c.A, user_base=c.user_base)
        dbg = nan(dev, N, D)
        kernels.score_fwd_tc(dims, dt['E_user'], PI, PF, gB, dt['expo'], dt['X'], dt['si'], rng, pred,
                             torch.empty(N, dtype=torch.float32, device=dev), dbg, err)
        out['dbg_pre'] = dbg
    else:
        save_h, save_w = nan(dev, N, D), nan(dev, P + extra, Z)
        kernels.score_fwd(dt['dims'], dt['E_user'], dt['E_item'], dt['Feat'], dt['W'], dt['b'], dt['expo'], dt['X'],
                          dt['si'], rng, pred, torch.empty(N, dtype=torch.float32, device=dev),
                          torch.empty((D + F) * D, dtype=torch.float32, device=dev), save_h, save_w, err)
        out['save_h'], out['save_w'] = save_h, save_w[:P]
        out['save_w_tail'] = save_w[P:]
    torch.cuda.synchronize()
    out['pred'], out['pred_tail'] = pred[:P], pred[P:]
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res['err'] = int(err[0])
    return res


def setup_scorer(c, dev):
    pb = make_scorer_problem(c)
    dt = _device_problem(pb, dev)
    M = None
    tables = gBp = None
    if c.scorer != 'simt':
        tables = prepare(dt, c.F, dev)
    if c.scorer == 'tc_projected':
        M = (np.random.RandomState(5).standard_normal((D, D)) * 0.1).astype(np.float32)
        gBp = projected_operand(M, dev)
    return pb, dt, tables, gBp, M


@pytest.mark.parametrize('name', [c.name for c in SCORER_CASES])
def test_scorer_equals_float64_reference(name):
    import torch
    c = SCASE[name]
    dev = torch.device('cuda:0')
    torch.cuda.set_device(0)
    pb, dt, tables, gBp, M = setup_scorer(c, dev)
    rng, noise, mask, keep = streams(c, pb, dev, D if c.scorer == 'tc_projected' else c.F)
    got, names = traced(lambda: run_scorer(c, dt, rng, dev, tables, gBp))
    assert got['err'] == 0
    assert launched(names, c.kernel), (c.kernel, sorted(names))
    if c.scorer != 'gather':
        assert launched(names, 'k_backdoor'), sorted(names)
    if c.scorer == 'simt':
        other = 'k_row_scores<' if 'splitk' in c.kernel else 'k_row_scores_splitk<'
        assert not any(other in n for n in names), sorted(names)
    ref, absv = scorer_reference(c, pb, noise, mask, M)
    if c.max_slots:
        # the softmax maximum first appears where the case put it (chunk 2 / 3 of the gather scorer)
        first = np.argmax(ref['w'], axis=1)
        assert np.array_equal(first, [c.max_slots[p % len(c.max_slots)] for p in range(c.P)])
    check_scorer(c, ref, absv, got)


@pytest.mark.parametrize('n_items,F', [(1, 64), (63, 768), (64, 1024), (65, 768), (65, 64)])
def test_tc_prepare_equals_float64_reference(n_items, F):
    """PI = E_item·W_i^T and PF = Feat·W_f^T + b element by element (the 64-row blocks of k_table_gemm, the second job
    starting in the block after the first's last); the W_f operand image: hi + lo == W_f exactly, hi = the top 19
    bits, lo = the exact remainder, every element where core_offset puts it."""
    import torch
    from dccf_b200 import kernels
    dev = torch.device('cuda:0')
    rs = np.random.RandomState(n_items * 7 + F)
    f32 = np.float32
    pb = {'E_user': np.zeros((4, D), f32), 'E_item': (rs.standard_normal((n_items, D)) * 0.05).astype(f32),
          'W': (rs.standard_normal((D, D + F)) * 0.05).astype(f32), 'b': (rs.standard_normal(D) * 0.05).astype(f32),
          'Feat': (rs.standard_normal((n_items, F)) / np.sqrt(F)).astype(f32), 'X': np.zeros((1, 2), np.int64),
          'si': np.zeros((1, 0), np.int64), 'expo': np.zeros((4, n_items), f32), 'F': F, 'S': 0, 'A': 1,
          'user_base': 0}
    dt = _device_problem(pb, dev)
    (PI, PF, gB), names = traced(lambda: prepare(dt, F, dev))
    for k in ('k_transpose_w', 'k_table_gemm', 'k_prep_wf'):
        assert launched(names, k), (k, sorted(names))
    W = pb['W'].astype(np.float64)
    E, Fe, b = pb['E_item'].astype(np.float64), pb['Feat'].astype(np.float64), pb['b'].astype(np.float64)
    ref = {'PI': E @ W[:, :D].T, 'PF': Fe @ W[:, D:].T + b}
    absv = {'PI': np.abs(E) @ np.abs(W[:, :D]).T, 'PF': np.abs(Fe) @ np.abs(W[:, D:]).T + np.abs(b)}
    got = {'PI': PI.cpu().numpy(), 'PF': PF.cpu().numpy()}
    fails, observed = compare(got, ref, c=C['prep'], bounds_fn=abs_bounds(absv), outputs=('PI', 'PF'))
    for k, v in observed.items():
        OBSERVED['prep', k] = max(OBSERVED['prep', k], v)
    print('prepare I=%d F=%d observed C: %s' % (n_items, F, ' '.join('%s %.3g' % kv for kv in observed.items())))
    assert not fails, fails
    img = gB.cpu().numpy()
    assert img.size == kernels.tc_operand_floats(F) == (F // TC_KC) * 4096
    idx = operand_index(F)
    hi, lo = img[idx], img[idx + 2048]
    Wf = np.ascontiguousarray(pb['W'][:, D:])
    assert not (hi.view(np.uint32) & np.uint32(0x1FFF)).any()
    assert np.array_equal(hi.view(np.uint32), tf32_hi(Wf).view(np.uint32))
    assert np.array_equal(hi.astype(np.float64) + lo.astype(np.float64), Wf.astype(np.float64))
    assert np.array_equal((hi + lo).view(np.uint32), Wf.view(np.uint32))


def _same_bits(x, y):
    x, y = np.asarray(x), np.asarray(y)
    return x.shape == y.shape and np.array_equal(x.reshape(-1).view(np.uint8), y.reshape(-1).view(np.uint8))


def test_scorer_bitwise_invariants():
    """Mode 2 (noise / mask generated in the kernel) equals mode 1 fed the materialised values, bit for bit, for the
    tensor-core and the SIMT scorer; two identical calls of every scorer give identical bits; an out-of-range id is
    reported through the error flag and nothing is written past n_pairs."""
    import torch
    dev = torch.device('cuda:0')
    for name in ('tc_f128_n2m2_r1', 'simt_37761', 'simt_r82', 'g_z41_p257'):
        c = SCASE[name]
        pb, dt, tables, gBp, M = setup_scorer(c, dev)
        rng, noise, mask, keep = streams(c, pb, dev, c.F)
        a = run_scorer(c, dt, rng, dev, tables, extra=5)
        b = run_scorer(c, dt, rng, dev, tables, extra=5)
        for k in a:
            assert _same_bits(a[k], b[k]), (name, k)
        if c.noise == 2 or c.mask == 2:
            rng1, _, _, keep1 = streams(c, pb, dev, c.F, materialised=True)
            assert rng1.noise_mode in (0, 1) and rng1.mask_mode in (0, 1)
            m1 = run_scorer(c, dt, rng1, dev, tables, extra=5)
            for k in a:
                assert _same_bits(a[k], m1[k]), (name, k)
        # an item id out of range in pair 1: flagged, and the buffers past n_pairs stay untouched
        if c.scorer in ('gather', 'simt'):
            bad = dict(pb)
            bad['X'], bad['si'] = pb['X'].copy(), pb['si'].copy()
            if c.S:
                bad['si'][min(1, c.P - 1), 0] = pb['Feat'].shape[0]
            else:
                bad['X'][min(1, c.P - 1), 1] = pb['Feat'].shape[0]
            dtb = _device_problem(bad, dev)
            e = run_scorer(c, dtb, rng, dev, tables, extra=5)
            assert e['err'] == 1, name
            assert np.isnan(e['pred_tail']).all(), name
            if 'save_w_tail' in e:
                assert np.isnan(e['save_w_tail']).all(), name


# ------------------------------------------------------------------------------------------------------------------
# the full-catalogue GEMM and its fused top-k
# ------------------------------------------------------------------------------------------------------------------
FCase = collections.namedtuple('FCase', 'name kind U I k excl')
FS_CASES = [
    FCase('u1_i1_k8', 'ipsmf', 1, 1, 8, False),                 # k > n_items: -1 padding
    FCase('u127_i31_k9_excl', 'dccf', 127, 31, 9, True),        # KCAP 16
    FCase('u128_i32_k16', 'ipsmf', 128, 32, 16, False),
    FCase('u129_i33_k8_excl', 'dccf', 129, 33, 8, True),        # KCAP 8
    FCase('u129_i64_k1_excl', 'ipsmf', 129, 64, 1, True),
    FCase('u128_i65_k9', 'dccf', 128, 65, 9, False),
    FCase('u127_i4097_k16_excl', 'ipsmf', 127, 4097, 16, True),  # 65 splits of one tile, a 1-item last tile
    FCase('u5000_i640_k8', 'ipsmf', 5000, 640, 8, False),        # 8 splits of 2 tiles for 10 tiles: 3 empty
    FCase('u5000_i640_k9_excl', 'dccf', 5000, 640, 9, True),
    FCase('u129_i4097_matrix', 'dccf', 129, 4097, 0, False),
]
FCASE = {c.name: c for c in FS_CASES}
DUP = 8       # items 0..7 repeated across both column halves of a tile and across item splits: exact ties


def dup_targets(I):
    return [t for t in (32, 64, 96, I - DUP) if t >= DUP and t + DUP <= I]


def make_fs_problem(c):
    """float32 operands of one case (the arrays dccf_full_scores reads) and the exclusion lists."""
    rs = np.random.RandomState(100 + FS_CASES.index(c) if c in FS_CASES else 7)
    f32 = np.float32
    A = (rs.standard_normal((c.U, D)) * 0.2).astype(f32)
    B = (rs.standard_normal((c.I, D)) * 0.2).astype(f32)
    p = {'A': A, 'B': B, 'rb': None, 'cb': None, 'cs': None, 'g': 0.0}
    if c.kind == 'ipsmf':
        p['rb'] = (rs.standard_normal(c.U) * 0.1).astype(f32)
        p['cb'] = (rs.standard_normal(c.I) * 0.1).astype(f32)
        p['cs'] = (1.0 / np.maximum(rs.uniform(0.01, 0.2, size=c.I).astype(f32), f32(0.0625))).astype(f32)
        p['g'] = 0.125
    else:
        p['B'] = np.maximum(B, 0).astype(f32)          # relu(PI + PF): the hidden vector of every item
    # item 0 leads every user's list; items 0..7 are duplicated: exact ties across halves and splits
    A[:, 0] += f32(1.0)
    p['B'][0, 0] += f32(3.0)
    for t in dup_targets(c.I):
        for key in ('B', 'cb', 'cs'):
            if p[key] is not None:
                p[key][t:t + DUP] = p[key][:DUP]
    lists = None
    if c.excl:
        lists = []
        for u in range(c.U):
            n = [0, 3, 40, c.I // 2][u % 4]
            n = min(n, c.I)
            l = sorted(rs.choice(c.I, size=n, replace=False).tolist())
            if u == 5 and c.I > 3:
                l = sorted(set(range(c.I)) - {0, c.I - 1})        # two rankable items: padded with -1
            if u == 6:
                l = [1, 2, 33] if c.I > 33 else [x for x in (1, 2) if x < c.I]      # one of the duplicated items
            lists.append(l)
    return p, lists


def fs_inputs(p):
    """The float32 values the kernel multiplies: fl(rb + g), fl(cs * B), cs, fl(cs * cb)."""
    f32 = np.float32
    if p['cs'] is None:
        return p['A'], p['B'], None, None, None
    rbg = (p['rb'] + f32(p['g'])).astype(f32)
    return p['A'], (p['B'] * p['cs'][:, None]).astype(f32), rbg, p['cs'], (p['cs'] * p['cb']).astype(f32)


def fs_reference(p, row_bias_after_scale=False):
    """(score [U, I], |score|_abs) in float64."""
    A, Bs, rbg, cs, cbs = (None if a is None else np.asarray(a, np.float64) for a in fs_inputs(p))
    ref = A @ Bs.T
    absv = np.abs(A) @ np.abs(Bs).T
    if cs is not None:
        if row_bias_after_scale:
            ref = ref + cbs[None, :] + rbg[:, None]
        else:
            ref = ref + rbg[:, None] * cs[None, :] + cbs[None, :]
        absv = absv + np.abs(rbg)[:, None] * np.abs(cs)[None, :] + np.abs(cbs)[None, :]
    return ref, absv


def fs_bound(ref, absv, c=None):
    return (C['fs']['scores'] if c is None else c) * UNIT * absv + ULPS * np.abs(ref)


def allowed_items(I, U, lists):
    return [np.arange(I) if lists is None else np.setdiff1d(np.arange(I), np.asarray(lists[u], np.int64))
            for u in range(U)]


def topk_of(M, k, allowed, desc_ties=False):
    """Top-k by (score desc, item id asc) over each row's allowed items; -1 / -inf padded."""
    U = M.shape[0]
    ids = -np.ones((U, k), np.int64)
    sc = np.full((U, k), -np.inf, np.float32)
    for u in range(U):
        cand = allowed[u]
        order = np.lexsort((-cand if desc_ties else cand, -M[u, cand].astype(np.float64)))[:k]
        top = cand[order]
        ids[u, :len(top)] = top
        sc[u, :len(top)] = M[u, top]
    return sc, ids


def check_topk(got_s, got_i, M_got, ref, bnd, k, allowed):
    """Failures of a fused top-k: (1) it is the exact top-k of the kernel's own scores (score desc, item id asc; so exact
    ties come out by ascending id across halves and splits) and its scores are those entries bit for bit; (2) its ids
    are the float64 order, except inside a run of candidates whose float64 scores lie within the sum of their
    bounds."""
    fails = []
    want_s, want_i = topk_of(M_got, k, allowed)
    if not np.array_equal(got_i, want_i):
        fails.append('top-k ids differ from the top-k of the kernel\'s own scores at %d places'
                     % int((got_i != want_i).sum()))
    if not np.array_equal(np.asarray(got_s, np.float32).view(np.uint32), want_s.view(np.uint32)):
        fails.append('top-k scores are not the matrix entries bit for bit')
    _, ref_i = topk_of(ref, k, allowed)
    bad = 0
    for u, t in np.argwhere(got_i != ref_i):
        g, r = got_i[u, t], ref_i[u, t]
        if g < 0 or r < 0 or abs(ref[u, g] - ref[u, r]) > bnd[u, g] + bnd[u, r]:
            bad += 1
    if bad:
        fails.append('%d top-k entries out of the float64 order beyond their bounds' % bad)
    return fails


def _csr(lists, dev):
    import torch
    off = np.zeros(len(lists) + 1, np.int64)
    off[1:] = np.cumsum([len(l) for l in lists])
    items = np.array([i for l in lists for i in l], np.int32)
    if items.size == 0:
        items = np.zeros(1, np.int32)
    return torch.from_numpy(off).to(dev), torch.from_numpy(items).to(dev)


def run_fs(p, dev, k, materialise, exclude=None):
    import torch
    from dccf_b200 import kernels
    t = {key: (None if p[key] is None else _t(p[key], dev)) for key in ('A', 'B', 'rb', 'cb', 'cs')}
    out = kernels.full_scores(t['A'], t['B'], t['rb'], t['cb'], t['cs'], p['g'], materialise=materialise, k=k,
                              exclude=exclude)
    torch.cuda.synchronize()
    return tuple(None if x is None else x.cpu().numpy() for x in out)


@pytest.mark.parametrize('name', [c.name for c in FS_CASES])
def test_full_scores_equal_float64_reference(name):
    import torch
    c = FCASE[name]
    dev = torch.device('cuda:0')
    torch.cuda.set_device(0)
    p, lists = make_fs_problem(c)
    ref, absv = fs_reference(p)
    # the matrix (with the unexcluded top-k in the same call when there is no exclusion)
    (M, ts, ti), names = traced(lambda: run_fs(p, dev, 0 if c.excl else c.k, True))
    assert launched(names, 'k_fs_prep_b') and launched(names, fs_kernel(0 if c.excl else c.k, False)), sorted(names)
    fails, observed = compare({'scores': M}, {'scores': ref}, c=C['fs'], bounds_fn=abs_bounds({'scores': absv}),
                              outputs=('scores',))
    OBSERVED['fs', 'scores'] = max(OBSERVED['fs', 'scores'], observed['scores'])
    print('%-22s splits %s observed C: scores %.3g' % (c.name, fs_geometry(c.U, c.I), observed['scores']))
    assert not fails, fails
    bnd = fs_bound(ref, absv)
    if c.k and not c.excl:
        assert launched(names, 'k_topk_merge')
        fails = check_topk(ts, ti, M, ref, bnd, c.k, allowed_items(c.I, c.U, None))
        assert not fails, fails
    if c.excl:
        (_, ts, ti), names = traced(lambda: run_fs(p, dev, c.k, False, exclude=_csr(lists, dev)))
        assert launched(names, fs_kernel(c.k, True)) and launched(names, 'k_topk_merge'), sorted(names)
        allowed = allowed_items(c.I, c.U, lists)
        fails = check_topk(ts, ti, M, ref, bnd, c.k, allowed)
        assert not fails, fails
        for u in range(c.U):
            assert not set(ti[u].tolist()) & set(lists[u])
    if c.k >= 2 and dup_targets(c.I):
        # duplicated items reach the lists: exact ties, broken by ascending id
        assert any(len(set(ts[u][ti[u] >= 0].tolist())) < int((ti[u] >= 0).sum()) for u in range(c.U))
    # two identical calls: identical bits
    M2 = run_fs(p, dev, 0, True)[0]
    assert np.array_equal(M.view(np.uint32), M2.view(np.uint32))


# ------------------------------------------------------------------------------------------------------------------
# DCCF.predict_many: the model's routing over a ragged evaluation set
# ------------------------------------------------------------------------------------------------------------------
def test_predict_many_equals_float64_reference():
    """Batches of N >= tc_min_rows rows go to the tensor-core scorer, the tail to k_row_scores_splitk, and at std = 0
    everything to the gather scorer; every prediction against the float64 reference on the noise rematerialised from
    the model's seed and the per-call offsets."""
    import torch
    from dccf_b200 import kernels
    from test_gpu_full_catalogue import _dccf
    torch.cuda.set_device(0)
    dev = torch.device('cuda:0')
    U, I, S = 60, 300, 10
    model = _dccf(U, I, S=S, std=STD)
    model.eval()
    A, F = model.attribute_num, model.feature_embedding.shape[1]
    R = (S + 1) * A
    sizes = [900, 900, 137]
    assert sizes[0] * R >= model.tc_min_rows > sizes[2] * R
    rs = np.random.RandomState(9)
    fds = [{'X': torch.from_numpy(np.stack([rs.randint(0, U, n), rs.randint(0, I, n)], 1)),
            'sample_item': torch.from_numpy(rs.randint(0, I, (n, S)))} for n in sizes]
    pb = {'E_user': model.uid_embeddings.weight.detach().cpu().numpy(),
          'E_item': model.iid_embeddings.weight.detach().cpu().numpy(),
          'W': model.mlp[0].weight.detach().cpu().numpy(), 'b': model.mlp[0].bias.detach().cpu().numpy(),
          'Feat': model.feature_embedding.cpu().numpy(), 'expo': model.expo_prob.cpu().numpy(),
          'F': F, 'S': S, 'A': A, 'user_base': 0}
    for std in (STD, 0.0):
        model.std = std
        off0 = model._rng_offset
        with torch.no_grad():
            outs, names = traced(lambda: [o.cpu().numpy() for o in model.predict_many(fds)])
        if std:
            assert launched(names, 'k_row_scores_tc<2>') and launched(names, 'k_row_scores_splitk<2>'), sorted(names)
            assert not launched(names, 'k_gather_scores')
        else:
            assert launched(names, 'k_gather_scores'), sorted(names)
            assert not any('k_row_scores' in n for n in names), sorted(names)
        for j, (fd, got) in enumerate(zip(fds, outs)):
            q = dict(pb, X=fd['X'].numpy(), si=fd['sample_item'].numpy())
            N = sizes[j] * R
            tc = std > 0 and N >= model.tc_min_rows
            noise = None
            if std:
                t = torch.empty((N, F), dtype=torch.float32, device=dev)
                noise = kernels.noise_fill(t, std, model.random_seed, off0 + j + 1).cpu().numpy()
            scorer = 'tc' if tc else ('simt' if std else 'gather')
            ref = forward_reference(q, noise, None, noise_exact=tc)
            fails, observed = compare({'pred': got}, ref, c=C[scorer], bounds_fn=fwd_bounds, outputs=('pred',))
            OBSERVED[scorer, 'pred'] = max(OBSERVED[scorer, 'pred'], observed['pred'])
            print('predict_many std %g batch %d (%s) observed C: pred %.3g' % (std, j, scorer, observed['pred']))
            assert not fails, (std, j, fails)


# ------------------------------------------------------------------------------------------------------------------
# the ranker's fallbacks
# ------------------------------------------------------------------------------------------------------------------
def ranker_problem(seed=3):
    """Users that reach every path of k_rank_stream: 2049 and 5000 candidates (past the staging buffer), 1001 equal
    scores, 129 candidates tied at the threshold behind three distinct leaders, all-NaN scores, an ordinary user."""
    rs = np.random.RandomState(seed)
    groups = []
    groups.append(rs.standard_normal(2049).astype(np.float32))
    s = rs.standard_normal(5000).astype(np.float32)
    s[100:200] = s[0]                                           # ties inside the long list
    groups.append(s)
    groups.append(np.full(1001, 0.25, np.float32))
    s = rs.uniform(-1.0, 0.4, 1001).astype(np.float32)
    s[rs.choice(1001, 129, replace=False)] = 0.5
    s[[3, 500, 900]] = [0.9, 0.8, 0.7]
    groups.append(s)
    groups.append(np.full(50, np.nan, np.float32))
    groups.append(rs.standard_normal(20).astype(np.float32))
    scores = np.concatenate(groups)
    uid = np.concatenate([np.full(len(g), u, np.int64) for u, g in enumerate(groups)])
    iids = np.concatenate([rs.permutation(10 ** 6)[:len(g)] for g in groups]).astype(np.int64)
    labels = (rs.uniform(size=len(scores)) < 0.05).astype(np.float32)
    off = np.zeros(len(groups) + 1, np.int64)
    off[1:] = np.cumsum([len(g) for g in groups])
    return scores, uid, labels, iids, off


def test_ranker_fallbacks_equal_the_oracle():
    import torch
    from dccf_b200 import kernels
    torch.cuda.set_device(0)
    scores, uid, labels, iids, off = ranker_problem()
    n_users = len(off) - 1
    sc, lb, ii, of = (torch.from_numpy(a).cuda() for a in (scores, labels, iids, off))
    ks = [1, 5, 16]
    per = torch.empty((n_users, len(ks), 5), dtype=torch.float64, device='cuda')
    topk = torch.empty((n_users, ks[-1]), dtype=torch.int64, device='cuda')
    _, names = traced(lambda: kernels.rank_eval_multi(sc, lb, ii, None, of, ks, out_metrics=per, out_topk_iid=topk))
    assert launched(names, 'k_rank_stream'), sorted(names)
    per, topk = per.cpu().numpy(), topk.cpu().numpy()
    for j, k in enumerate(ks):
        _, want_ids, _, want_m = O.rank_users(scores, uid, labels, iids, k)
        assert np.array_equal(topk[:, :k], want_ids), k
        assert np.array_equal(np.isnan(per[:, j]), np.isnan(want_m)), k
        assert np.nanmax(np.abs(per[:, j] - want_m)) <= 1e-12, k
    k = 20
    m = torch.empty((n_users, 5), dtype=torch.float64, device='cuda')
    ids = torch.empty((n_users, k), dtype=torch.int64, device='cuda')
    _, names = traced(lambda: kernels.rank_eval(sc, lb, ii, None, of, k, m, out_topk_iid=ids))
    assert launched(names, 'k_rank_select'), sorted(names)
    _, want_ids, _, want_m = O.rank_users(scores, uid, labels, iids, k)
    m = m.cpu().numpy()
    assert np.array_equal(ids.cpu().numpy(), want_ids)
    assert np.array_equal(np.isnan(m), np.isnan(want_m))
    assert np.nanmax(np.abs(m - want_m)) <= 1e-12
