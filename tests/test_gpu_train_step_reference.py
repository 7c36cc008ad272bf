"""Every output of one call of the tensor-core training step (dccf_train_fwd_bwd_tc), and of the two pairs of calls it
falls back to (the unfused tensor-core pair dccf_train_fwd_tc + dccf_train_bwd_tc, the SIMT pair dccf_score_fwd +
dccf_bpr_bwd), against a float64 reference (oracle/dccf_oracle.py), element by element, over the step's launch
geometry: K splits 1 to 8, feature widths with and without a bias-only last M tile of the dW kernel, single- and
multi-pass phases of the middle kernel, both sides of its shared-memory limit, every noise / dropout mode, BPR and MSE,
dense and IPS-MF exposure, a user shard (user_base != 0) and a wide-range problem.  Then the bitwise invariants of the
step (phase splits, programmatic launches, precomputed exposure softmax, the device-side RNG offset) and the step on a
second GPU of the same process.

Tolerance.  Element y of an output must satisfy |y_kernel - y_ref| <= C * 2^-20 * |y|_abs + (a few ulps), where |y|_abs
is the same computation run on absolute values (|x| @ |W|^T for the pre-activations, |dpre|^T @ |x| for gW, ...) and
the bound of each stage's inputs is carried through it to first order (softmax, loss, records).  The bound is affine in
C, so `observed` reports the smallest C each output needs; C is about four times the largest one seen on a B200.
Pre-activations within their own bound of zero may gate the other way in the kernel (the ReLU kink): for those, and
only those, the reference takes the gate from the kernel's save_h; everywhere else the gates must agree exactly."""
import collections

import numpy as np
import pytest

from oracle import dccf_oracle as O

pytestmark = pytest.mark.gpu

D = 64
TC_BM, TC_KC, N_SM = 128, 32, 148        # tile rows, K chunk width, SMs the heuristics size the grids for
FUSED_SMEM_LIMIT = 200 * 1024
UNIT = 2.0 ** -20
C = 0.875                                 # 4 x 0.213, the largest ratio observed on a B200 (save_h, ks1_p512)
ULPS = 8 * 2.0 ** -24                     # the few ulps of |y| every bound carries (rounding of the output itself)
STD, P_DROP = 0.1, 0.2


# ------------------------------------------------------------------------------------------------------------------
# the launch geometry, mirrored from tc_train.cu (fwd_ksplits_for, bwd_geometry, train_mid_smem_floats) and bpr_bwd.cu
# (bwd_splits_for at the reference chunk count); tests/test_train_step_reference_cpu.py pins them to the library
# ------------------------------------------------------------------------------------------------------------------
def fwd_ksplits_for(n_rows, F):
    if n_rows <= 0:
        return 1
    tiles = -(-n_rows // TC_BM)
    return max(1, min(N_SM // tiles, 8, (D + F) // TC_KC))


def bwd_geometry(n_rows, F):
    """(M tiles of [x | 1], row splits, rows per split) of the dW kernel."""
    mt = -(-(D + F + 1) // TC_BM)
    want = max(N_SM // mt, 1)
    rps = max(-(-(-(-n_rows // want)) // TC_KC) * TC_KC, TC_KC)
    return mt, max(-(-n_rows // rps), 1), rps


def simt_geometry(n_rows):
    """(row splits, rows per split) of k_bpr_bwd's gW role."""
    ns = 1 if n_rows <= 0 else max(1, min(-(-2 * N_SM // 13), -(-n_rows // 64)))
    rps = -(-n_rows // ns)
    return ns, -(-rps // 16) * 16


def mid_smem_bytes(S, A, loss_mode):
    Z = S + 1
    R, npc = Z * A, (2 if loss_mode == 0 else 1)
    return 4 * (D * D + npc * R * D + npc * Z * D + npc * R + npc * Z + 8)


def split_rows(n_rows, n_splits, rps):
    return [(sp * rps, min((sp + 1) * rps, n_rows)) for sp in range(n_splits)]


# ------------------------------------------------------------------------------------------------------------------
# cases: one list; each states the geometry it is meant to reach (checked against the library before it runs)
# ------------------------------------------------------------------------------------------------------------------
Case = collections.namedtuple('Case', 'name F P S A loss noise mask expo user_base mse_pairs wide paths ks splits fused')
CASES = [
    # F=64: 4 K chunks, every one its own split (ks = n_chunks); S=0, A=1; BPR with one loss term
    Case('bpr_p2_s0a1', 64, 2, 0, 1, 0, 0, 0, 'dense', 0, 0, False, ('fused', 'simt'), 4, 1, True),
    # the default shape: 44 row tiles, 3 K splits, 20 row splits of the dW kernel
    Case('default', 768, 256, 10, 2, 0, 2, 2, 'dense', 0, 0, False, ('fused', 'tc', 'simt'), 3, 20, True),
    # 88 row tiles: one K split; P >= 512
    Case('ks1_p512', 1024, 512, 10, 2, 0, 1, 1, 'dense', 0, 0, False, ('fused',), 1, 16, True),
    # 52 row tiles: 2 K splits; A=3: phase A of the middle kernel takes two passes (2 x 33 rows)
    Case('ks2_s10a3', 384, 200, 10, 3, 0, 2, 1, 'ipsmf', 0, 0, False, ('fused',), 2, 35, True),
    # 26 row tiles: 5 K splits; S=40: C1 / C2 multi-pass, 80 KB of shared memory (opt-in); K+1 = 257: bias-only M tile
    Case('ks5_s40a2', 192, 40, 40, 2, 0, 1, 2, 'dense', 0, 0, False, ('fused', 'tc'), 5, 35, True),
    # 8 K splits; S=119, A=2: 203 616 B, the largest fused middle kernel at A=2; K+1 = 1025: bias-only M tile
    Case('ks8_s119a2', 960, 4, 119, 2, 0, 2, 0, 'ipsmf', 0, 0, False, ('fused',), 8, 15, True),
    # S=120, A=2: past the fused limit, the unfused pair
    Case('s120a2_unfused', 2048, 4, 120, 2, 0, 0, 1, 'dense', 0, 0, False, ('tc', 'simt'), 8, 8, False),
    # S=180, A=1: 204 656 B, still fused; a user shard
    Case('s180a1', 768, 6, 180, 1, 0, 1, 0, 'ipsmf', 1000, 0, False, ('fused',), 8, 17, True),
    # S=181, A=1: falls back
    Case('s181a1_unfused', 64, 4, 181, 1, 0, 2, 2, 'dense', 0, 0, False, ('tc', 'simt'), 4, 23, False),
    # MSE with one pair
    Case('mse_p1', 192, 1, 10, 2, 1, 0, 2, 'dense', 0, 0, False, ('fused', 'tc'), 8, 1, True),
    # MSE with three pairs, a mean over 7 (a data-parallel step's count), a user shard, IPS-MF exposure
    Case('mse_p3_shard', 384, 3, 10, 3, 1, 1, 1, 'ipsmf', 17, 7, False, ('fused', 'simt'), 8, 4, True),
    # columns of E_item / Feat scaled by 2^-6 / 2^6, exposure over 35 nats (exp overflows without the max subtraction)
    Case('wide_range', 768, 64, 10, 2, 0, 2, 2, 'wide', 0, 0, True, ('fused', 'tc'), 8, 15, True),
    # 60 row splits of 32 rows, the last one 2 rows; ks = n_chunks; A=3 multi-pass phase A
    Case('splits60_last2', 64, 42, 14, 3, 0, 2, 1, 'dense', 0, 0, False, ('fused', 'simt'), 4, 60, True),
]
CASE = {c.name: c for c in CASES}


def n_rows_of(case):
    return case.P * (case.S + 1) * case.A


def make_problem(case, seed=0):
    """float32 / int64 host arrays of one case (global user ids in X when user_base != 0)."""
    rs = np.random.RandomState(1000 + seed + 7 * CASES.index(case) if case in CASES else seed)
    F, P, S, A = case.F, case.P, case.S, case.A
    U, I = 37, 211
    K, N = D + F, n_rows_of(case)
    f32 = np.float32
    pb = {'F': F, 'S': S, 'A': A, 'loss': case.loss, 'user_base': case.user_base,
          'E_user': (rs.standard_normal((U, D)) * 0.05).astype(f32),
          'E_item': (rs.standard_normal((I, D)) * 0.05).astype(f32),
          'W': (rs.standard_normal((D, K)) * 0.05).astype(f32),
          'b': (rs.standard_normal(D) * 0.05).astype(f32),
          'Feat': (rs.standard_normal((I, F)) / np.sqrt(F)).astype(f32)}
    if case.wide:
        scale = 2.0 ** rs.choice([-6, 0, 6], size=K)
        pb['E_item'] = (pb['E_item'] * scale[:D]).astype(f32)
        pb['Feat'] = (pb['Feat'] * scale[D:]).astype(f32)
    if case.expo == 'ipsmf':
        pb['ipsmf'] = {'mf_user': (rs.standard_normal((U, D)) * 0.2).astype(f32),
                       'mf_item': (rs.standard_normal((I, D)) * 0.2).astype(f32),
                       'mf_user_bias': (rs.standard_normal(U) * 0.1).astype(f32),
                       'mf_item_bias': (rs.standard_normal(I) * 0.1).astype(f32),
                       # about a third of the items below the floor
                       'propensity': rs.uniform(0.01, 0.2, size=I).astype(f32),
                       'mf_global_bias': 0.125, 'mf_min_propensity': 0.0625}
    elif case.expo == 'wide':
        pb['expo'] = rs.uniform(60.0, 95.0, size=(U, I)).astype(f32)
    else:
        pb['expo'] = rs.uniform(0.0, 1.0, size=(U, I)).astype(f32)
    if case.loss == 0:
        b = P // 2
        u = rs.randint(0, U, size=b)
        X = np.concatenate([np.stack([u, rs.randint(0, I, size=b)], 1), np.stack([u, rs.randint(0, I, size=b)], 1)])
    else:
        X = np.stack([rs.randint(0, U, size=P), rs.randint(0, I, size=P)], 1)
        pb['Y'] = rs.uniform(1.0, 5.0, size=P).astype(f32)
    X = X.astype(np.int64)
    X[:, 0] += case.user_base
    pb['X'] = X
    pb['si'] = rs.randint(0, I, size=(P, S)).astype(np.int64)
    if case.noise == 1:
        pb['noise'] = (rs.standard_normal((N, F)) * STD).astype(f32)
    if case.mask == 1:
        pb['mask'] = ((rs.uniform(size=(N, D)) < 1 - P_DROP) / (1 - P_DROP)).astype(f32)
    return pb


# ------------------------------------------------------------------------------------------------------------------
# float64 reference and its elementwise bounds
# ------------------------------------------------------------------------------------------------------------------
def forward_reference(pb, noise, mask, save_h=None, c=C, W=None, b=None, noise_exact=False):
    """float64 value of the forward (pre, h, w, s, pred) and what its bound is made of.  noise / mask: the float32
    values the kernels use (None: mode 0); save_h: the kernel's activations, which decide the gates of the kink
    elements.  W / b override pb's (the comparator's negative controls).  noise_exact: the kernel multiplies eps itself
    into W_f (the tensor-core scorer) instead of the rounded sum fl(Feat + eps)."""
    S, A, F = pb['S'], pb['A'], pb['F']
    Z = S + 1
    R = Z * A
    X = pb['X'].copy()
    X[:, 0] -= pb['user_base']
    P = X.shape[0]
    N = P * R
    params = {k: pb[k].astype(np.float64) for k in ('E_user', 'E_item', 'W', 'b', 'Feat')}
    if W is not None:
        params['W'] = W.astype(np.float64)
    if b is not None:
        params['b'] = b.astype(np.float64)
    expo = None
    if 'ipsmf' in pb:
        expo = {k: (np.asarray(v, np.float64) if not isinstance(v, float) else v) for k, v in pb['ipsmf'].items()}
    else:
        params['expo'] = pb['expo'].astype(np.float64)
    noise_eff = None
    if noise is not None:
        # the kernels add the noise in float32: x = fl(Feat + eps), which the oracle then sees exactly
        feat = pb['Feat'][np.repeat(X[:, 1], R)]
        noise_eff = noise.astype(np.float64) if noise_exact else \
            (feat + noise).astype(np.float64) - feat.astype(np.float64)
    m = np.ones((N, D)) if mask is None else mask.astype(np.float64)
    fwd = O.predict(params, X, pb['si'], noise_eff, None if mask is None else m, A, dtype=np.float64, expo=expo)
    x, pre, h, w, items = fwd['x'], fwd['pre'], fwd['h'], fwd['w'], fwd['items']
    u = X[:, 0]

    absP = np.abs(x) @ np.abs(params['W']).T + np.abs(params['b'])
    kink = (np.abs(pre) <= c * UNIT * absP) & (m != 0)
    gpos = pre > 0
    if save_h is not None:
        gpos = np.where(kink, save_h > 0, gpos)
    gv = gpos * m                                # d h / d pre
    live = (pre > 0) | kink                      # elements whose h may be non-zero in the kernel

    v = O.exposure_values(expo if expo is not None else params['expo'], u, items)
    if expo is not None:
        v_abs = (np.einsum('pd,pzd->pz', np.abs(expo['mf_user'][u]), np.abs(expo['mf_item'][items]))
                 + np.abs(expo['mf_user_bias'][u])[:, None] + np.abs(expo['mf_item_bias'][items])
                 + abs(expo['mf_global_bias'])) / np.maximum(expo['propensity'][items], expo['mf_min_propensity'])
    else:
        v_abs = np.zeros_like(v)
    rho = 1.0 + np.abs(v - v.max(axis=1, keepdims=True)) + v_abs + v_abs.max(axis=1, keepdims=True)
    return {'P': P, 'Z': Z, 'R': R, 'A': A, 'N': N, 'x': x, 'pre': pre, 'h': h, 'w': w, 's': fwd['s'],
            'pred': fwd['pred'], 'save_h': h, 'save_w': w, 'm': m, 'absP': absP, 'kink': kink, 'gpos': gpos, 'gv': gv,
            'live': live, 'rho': rho, 'eu_r': np.repeat(params['E_user'][u], R, axis=0), 'fwd': fwd, 'params': params,
            'X': X, 'noise_eff': noise_eff, 'items': items, 'u': u}


def reference(pb, noise, mask, mse_pairs, splits, save_h=None, c=C, W=None, b=None):
    """float64 value of every output of one step, and what its bound is made of.  noise / mask: the float32 values the
    kernels use (None: mode 0); mse_pairs: the MSE divisor; splits: [(row_lo, row_hi)] of the gW / gb partials;
    save_h: the kernel's activations, which decide the gates of the kink elements.  W / b override pb's in the forward
    only (the comparator's negative controls)."""
    ref = forward_reference(pb, noise, mask, save_h=save_h, c=c, W=W, b=b)
    P, Z, R, A, N = ref['P'], ref['Z'], ref['R'], ref['A'], ref['N']
    x, h, w, pred, gv, eu_r, u = ref['x'], ref['h'], ref['w'], ref['pred'], ref['gv'], ref['eu_r'], ref['u']
    W64 = pb['W'].astype(np.float64)            # the backward's W (gi) is always the step's own

    if pb['loss'] == 0:
        hb = P // 2
        d = pred[:hb] - pred[hb:]
        sig = 1.0 / (1.0 + np.exp(-d))
        g = -(1.0 - sig)
        dp = np.concatenate([g, -g])
        loss = float(np.sum(np.logaddexp(0.0, -d)))
    else:
        d = pred - pb['Y'].astype(np.float64)
        sig = g = None
        dp = 2.0 * d / mse_pairs
        loss = float(np.sum(d * d) / mse_pairs)
    ds = dp[:, None] * w / A                                                   # [P, Z]
    ds_r = np.repeat(ds.reshape(-1), A)                                        # [N]
    dpre = ds_r[:, None] * eu_r * gv
    gu = (ds_r[:, None] * h).reshape(P, R, D).sum(axis=1)
    gi = (dpre.reshape(P, Z, A, D).sum(axis=2) @ W64[:, :D]).reshape(P * Z, D)
    gW = np.stack([dpre[lo:hi].T @ x[lo:hi] for lo, hi in splits])
    gb = np.stack([dpre[lo:hi].sum(axis=0) for lo, hi in splits])

    ref.update({'loss_mode': pb['loss'], 'd': d, 'sig': sig, 'g': g, 'dp': dp, 'mse_pairs': mse_pairs, 'loss': loss,
                'ds': ds, 'ds_r': ds_r, 'dpre': dpre, 'gu': gu, 'gi': gi, 'gW': gW, 'gb': gb, 'W': W64,
                'splits': splits, 'ku': u.astype(np.int32), 'ki': ref['items'].reshape(-1).astype(np.int32)})
    return ref


def forward_bounds(ref, eps):
    """Elementwise error bounds of the forward's outputs (save_h, save_w, pred) for a relative unit eps (= C * 2^-20),
    first order: each stage's bound is eps times its absolute-value computation, plus its inputs' bounds carried
    through it, plus ULPS of the value.  Also returns the bound of the row scores (Bs) and the softmax's relative
    bound (rel_w), which the backward's bounds carry on."""
    P, R, A = ref['P'], ref['R'], ref['A']
    h, w, s, m, eu_r = ref['h'], ref['w'], ref['s'], ref['m'], ref['eu_r']
    aeu = np.abs(eu_r)
    B = {}
    Bh = eps * ref['absP'] * np.abs(m) * ref['live'] + ULPS * np.abs(h)
    B['save_h'] = Bh
    Bs = (Bh * aeu).sum(axis=1) + eps * (np.abs(h) * aeu).sum(axis=1)                       # [N] row scores
    rho = ref['rho']
    rel_w = eps * (rho + (w * rho).sum(axis=1, keepdims=True) + 1.0)                        # softmax, relative
    B['save_w'] = rel_w * w + ULPS * w
    wr = np.repeat(w / A, A, axis=1)                                                        # [P, R]
    sr = np.abs(s.reshape(P, R))
    B['pred'] = (wr * (Bs.reshape(P, R) + sr * np.repeat(rel_w, A, axis=1))).sum(axis=1) \
        + eps * (wr * sr).sum(axis=1) + ULPS * np.abs(ref['pred'])
    return B, Bs, rel_w


def bounds(ref, eps):
    """Elementwise error bounds of every output for a relative unit eps (= C * 2^-20), first order: each stage's bound
    is eps times its absolute-value computation, plus its inputs' bounds carried through it, plus ULPS of the value."""
    P, Z, R, A, N = ref['P'], ref['Z'], ref['R'], ref['A'], ref['N']
    h, w, s, m, eu_r = ref['h'], ref['w'], ref['s'], ref['m'], ref['eu_r']
    aeu = np.abs(eu_r)
    B, Bs, rel_w = forward_bounds(ref, eps)
    Bh, Bw, Bpred = B['save_h'], B['save_w'], B['pred']
    dp = ref['dp']
    if ref['loss_mode'] == 0:
        hb = P // 2
        sig, g, d = ref['sig'], ref['g'], ref['d']
        Bd = Bpred[:hb] + Bpred[hb:]
        Bg = sig * (1 - sig) * Bd + ULPS * (np.abs(g) + sig)
        Bdp = np.concatenate([Bg, Bg])
        term = np.logaddexp(0.0, -d)
        B['loss'] = float(((1 - sig) * Bd + ULPS * term).sum() + eps * term.sum())
    else:
        M, d = ref['mse_pairs'], ref['d']
        Bdp = 2 * Bpred / M + ULPS * np.abs(dp)
        B['loss'] = float((2 * np.abs(d) * Bpred).sum() / M + eps * (d * d).sum() / M + ULPS * ref['loss'])
    ds = ref['ds']
    Bds = (Bdp[:, None] * w + np.abs(dp)[:, None] * Bw) / A + ULPS * np.abs(ds)
    Bds_r = np.repeat(Bds.reshape(-1), A)
    ads_r = np.abs(ref['ds_r'])
    dpre = ref['dpre']
    adpre = np.abs(dpre)
    Bdpre = Bds_r[:, None] * aeu * np.abs(ref['gv']) + ULPS * adpre
    B['dpre'] = Bdpre
    B['gu'] = ((Bds_r[:, None] * np.abs(h) + ads_r[:, None] * Bh).reshape(P, R, D).sum(axis=1)
               + eps * (ads_r[:, None] * np.abs(h)).reshape(P, R, D).sum(axis=1) + ULPS * np.abs(ref['gu']))
    aWi = np.abs(ref['W'][:, :D])
    B['gi'] = ((Bdpre.reshape(P, Z, A, D).sum(axis=2) @ aWi + eps * (adpre.reshape(P, Z, A, D).sum(axis=2) @ aWi))
               .reshape(P * Z, D) + ULPS * np.abs(ref['gi']))
    ax = np.abs(ref['x'])
    B['gW'] = np.stack([Bdpre[lo:hi].T @ ax[lo:hi] + eps * (adpre[lo:hi].T @ ax[lo:hi]) for lo, hi in ref['splits']]) \
        + ULPS * np.abs(ref['gW'])
    B['gb'] = np.stack([Bdpre[lo:hi].sum(axis=0) + eps * adpre[lo:hi].sum(axis=0) for lo, hi in ref['splits']]) \
        + ULPS * np.abs(ref['gb'])
    return B


OUTPUTS = ('pred', 'loss', 'save_h', 'save_w', 'dpre', 'gu', 'gi', 'gW', 'gb')


def compare(got, ref, c=C, bounds_fn=bounds, outputs=OUTPUTS):
    """got: numpy outputs of one call (any subset of `outputs`, plus 'ku' / 'ki').  Returns (failures, observed): the
    list of failed checks (empty = pass) and, per output, the smallest C its elements need (inf: an element that must
    be exact is not).  c: one C for every output or a dict of them; bounds_fn(ref, eps) -> {output: bound}."""
    B0 = bounds_fn(ref, 0.0)
    B1 = bounds_fn(ref, UNIT)
    fails, observed = [], {}
    for k in outputs:
        if k not in got:
            continue
        ck = c[k] if isinstance(c, dict) else c
        y = np.asarray(got[k], np.float64)
        r = np.asarray(ref[k], np.float64)
        if y.shape != r.shape:
            fails.append('%s: shape %s, reference %s' % (k, y.shape, r.shape))
            continue
        b0 = np.asarray(B0[k], np.float64)
        slope = np.asarray(B1[k], np.float64) - b0
        err = np.abs(y - r)
        err = np.where(np.isfinite(y), err, np.inf)
        excess = err - b0
        need = np.where(excess <= 0, 0.0, np.where(slope > 0, excess / np.where(slope > 0, slope, 1.0), np.inf))
        observed[k] = float(need.max()) if need.size else 0.0
        bad = ~(err <= b0 + ck * slope)
        if bad.any():
            i = np.unravel_index(int(np.argmax(np.where(bad, need, -1.0))), y.shape) if y.ndim else ()
            fails.append('%s: %d of %d elements outside the bound; worst at %s: kernel %r, reference %r, bound %.3g '
                         '(needs C = %.3g)' % (k, int(bad.sum()), bad.size, tuple(int(t) for t in i), float(y[i]),
                                               float(r[i]), float(b0[i] + ck * slope[i]), float(need[i])))
    for k in ('ku', 'ki'):
        if k in got and not np.array_equal(np.asarray(got[k]), ref[k]):
            fails.append('%s: record keys differ at %d places' % (k, int((np.asarray(got[k]) != ref[k]).sum())))
    if 'save_h' in got:
        # outside the kink the kernel gates exactly as the reference (where the dropout mask keeps the element)
        keep = (ref['m'] != 0) & ~ref['kink']
        flips = int(((np.asarray(got['save_h']) > 0) != (ref['pre'] > 0))[keep].sum())
        if flips:
            fails.append('gates: %d ReLU gates differ from the reference on elements outside the kink' % flips)
    return fails, observed


def cross_check_with_oracle(ref, pb, mask):
    """The in-module backward equals oracle.backward (the pinned restatement of autograd) on the same patched gates."""
    fwd = dict(ref['fwd'])
    fwd['pre'] = np.where(ref['gpos'], 1.0, -1.0)
    scale = 1.0 if ref['loss_mode'] == 0 else ref['P'] / ref['mse_pairs']
    gr = O.backward(ref['params'], ref['X'], pb['si'], ref['noise_eff'], None if mask is None else ref['m'], ref['A'],
                    fwd, loss_mode=ref['loss_mode'], Y=pb.get('Y'), dtype=np.float64)
    for k, mine in (('gu_rows', ref['gu']), ('gi_rows', ref['gi']), ('W', ref['gW'].sum(axis=0)),
                    ('b', ref['gb'].sum(axis=0))):
        theirs = gr[k] * scale
        assert np.allclose(mine, theirs, rtol=1e-10, atol=1e-12 * max(1e-300, np.abs(theirs).max())), k


# ------------------------------------------------------------------------------------------------------------------
# running the kernels
# ------------------------------------------------------------------------------------------------------------------
def _device_problem(pb, dev):
    import torch
    from dccf_b200 import kernels

    def t(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dt = {k: t(pb[k]) for k in ('E_user', 'E_item', 'W', 'b', 'Feat', 'X', 'si')}
    dt['Y'] = t(pb['Y']) if 'Y' in pb else None
    if 'ipsmf' in pb:
        dt['ipsmf'] = {k: (t(v) if isinstance(v, np.ndarray) else v) for k, v in pb['ipsmf'].items()}
        dt['expo'] = kernels.make_expo(ipsmf=dt['ipsmf'])
    else:
        dt['dense'] = t(pb['expo'])
        dt['expo'] = kernels.make_expo(dense=dt['dense'])
    dt['dims'] = kernels.make_dims(pb['E_user'].shape[0], pb['E_item'].shape[0], pb['F'], pb['S'], pb['A'],
                                   user_base=pb['user_base'])
    return dt


def _rng(case, pb, dt, dev, seed=2019, offset=5, offset_dev=False):
    """(rng struct, noise values, mask values) of the case; mode 2 values from the library's materialisers."""
    import torch
    from dccf_b200 import kernels
    N, F = n_rows_of(case), case.F
    noise = mask = None
    if case.noise == 1:
        dt['noise'] = torch.from_numpy(pb['noise']).to(dev)
        noise = pb['noise']
    elif case.noise == 2:
        t = torch.empty((N, F), dtype=torch.float32, device=dev)
        kernels.noise_fill(t, STD, seed, offset)
        noise = t.cpu().numpy()
    if case.mask == 1:
        dt['mask'] = torch.from_numpy(pb['mask']).to(dev)
        mask = pb['mask']
    elif case.mask == 2:
        t = torch.empty((N, D), dtype=torch.float32, device=dev)
        kernels.dropout_mask_fill(t, P_DROP, seed, offset)
        mask = t.cpu().numpy()
    if offset_dev:
        dt['offset_dev'] = torch.full((1,), offset, dtype=torch.int64, device=dev)
    rng = kernels.make_rng(noise=dt.get('noise'), mask=dt.get('mask'), noise_std=STD, p_drop=P_DROP, seed=seed,
                           offset=0 if offset_dev else offset, offset_dev=dt.get('offset_dev'),
                           generate_noise=case.noise == 2, generate_mask=case.mask == 2)
    return rng, noise, mask


def _buffers(case, dev, n_splits):
    import torch
    P, Z, N, K = case.P, case.S + 1, n_rows_of(case), D + case.F

    def nan(*shape):     # unwritten elements fail the comparison
        return torch.full(shape, float('nan'), dtype=torch.float32, device=dev)

    def keys(n):
        return torch.full((n,), -7, dtype=torch.int32, device=dev)
    return {'pred': nan(P), 'loss': nan(1), 'save_h': nan(N, D), 'save_w': nan(P, Z), 'dpre': nan(N, D),
            'gW': nan(n_splits, D, K), 'gb': nan(n_splits, D), 'gu': nan(P, D), 'gi': nan(P * Z, D),
            'ku': keys(P), 'ki': keys(P * Z), 'err': torch.zeros(1, dtype=torch.int32, device=dev)}


def _host(bufs, names):
    import torch
    torch.cuda.synchronize()
    assert int(bufs['err'][0]) == 0, 'the kernels flagged an id out of range'
    out = {k: bufs[k].cpu().numpy() for k in names}
    out['loss'] = float(bufs['loss'][0])
    return out


def run_fused(case, dt, rng, dev, calls=((7, False),), expo_split=False, batch=None):
    """dccf_train_fwd_bwd_tc, as one call or several (phases, w_image_valid) calls on the same buffers."""
    import torch
    from dccf_b200 import kernels
    N, F, P = n_rows_of(case), case.F, case.P
    bufs = _buffers(case, dev, kernels.train_bwd_splits(N, F))
    wimg = torch.empty(kernels.train_w_image_floats(F), dtype=torch.float32, device=dev)
    pre_part = torch.empty((kernels.train_fwd_ksplits(N, F), N, D), dtype=torch.float32, device=dev)
    terms = torch.empty(P // 2 if case.loss == 0 else P, dtype=torch.float32, device=dev)
    expo_e = expo_den = None
    if expo_split:
        Z = case.S + 1
        expo_e = torch.empty((P, Z), dtype=torch.float32, device=dev)
        expo_den = torch.empty(P, dtype=torch.float32, device=dev)
        head_u = torch.full((dt['E_user'].shape[0],), -1, dtype=torch.int32, device=dev)
        head_i = torch.full((dt['E_item'].shape[0],), -1, dtype=torch.int32, device=dev)
        next_u = torch.empty(P, dtype=torch.int32, device=dev)
        next_i = torch.empty(P * Z, dtype=torch.int32, device=dev)
        kernels.adam_link_ids(dt['dims'], dt['X'], dt['si'], head_u, next_u, head_i, next_i, dt['expo'], expo_e,
                              expo_den)
    for phases, w_valid in calls:
        if w_valid:
            kernels.train_prep_w_image(dt['W'], F, wimg)
        kernels.train_fwd_bwd_tc(dt['dims'], dt['E_user'], dt['E_item'], dt['Feat'], dt['W'], dt['b'], dt['expo'],
                                 dt['X'], dt['si'], dt['Y'], rng, case.loss, bufs['pred'], bufs['loss'], wimg, w_valid,
                                 pre_part, bufs['dpre'], terms, bufs['gW'], bufs['gb'], bufs['gu'], bufs['gi'],
                                 bufs['ku'], bufs['ki'], bufs['save_h'], bufs['save_w'], expo_e, expo_den,
                                 err_flag=bufs['err'], phases=phases, batch=batch, mse_pairs=case.mse_pairs)
    return _host(bufs, ('pred', 'save_h', 'save_w', 'dpre', 'gW', 'gb', 'gu', 'gi', 'ku', 'ki'))


def run_tc_pair(case, dt, rng, dev):
    """dccf_train_fwd_tc + dccf_train_bwd_tc: the production path beyond the fused limit."""
    import torch
    from dccf_b200 import kernels
    N, F = n_rows_of(case), case.F
    bufs = _buffers(case, dev, kernels.train_bwd_splits(N, F))
    ws_rows = torch.empty(N, dtype=torch.float32, device=dev)
    wimg = torch.empty(kernels.train_w_image_floats(F), dtype=torch.float32, device=dev)
    pre_part = torch.empty((kernels.train_fwd_ksplits(N, F), N, D), dtype=torch.float32, device=dev)
    kernels.train_fwd_tc(dt['dims'], dt['E_user'], dt['E_item'], dt['Feat'], dt['W'], dt['b'], dt['expo'], dt['X'],
                         dt['si'], rng, bufs['pred'], ws_rows, wimg, pre_part, bufs['save_h'], bufs['save_w'],
                         bufs['err'])
    kernels.train_bwd_tc(dt['dims'], dt['E_user'], dt['E_item'], dt['Feat'], dt['W'], dt['X'], dt['si'], dt['Y'], rng,
                         case.loss, bufs['pred'], bufs['save_h'], bufs['save_w'], bufs['loss'], bufs['gW'], bufs['gb'],
                         bufs['gu'], bufs['gi'], bufs['ku'], bufs['ki'], bufs['dpre'])
    return _host(bufs, ('pred', 'save_h', 'save_w', 'dpre', 'gW', 'gb', 'gu', 'gi', 'ku', 'ki'))


def run_simt(case, dt, rng, dev):
    """dccf_score_fwd + dccf_bpr_bwd (FP32 SIMT)."""
    import torch
    from dccf_b200 import kernels
    N, K = n_rows_of(case), D + case.F
    bufs = _buffers(case, dev, kernels.bwd_splits(N))
    ws_rows = torch.empty(N, dtype=torch.float32, device=dev)
    ws_wt = torch.empty(K * D, dtype=torch.float32, device=dev)
    kernels.score_fwd(dt['dims'], dt['E_user'], dt['E_item'], dt['Feat'], dt['W'], dt['b'], dt['expo'], dt['X'],
                      dt['si'], rng, bufs['pred'], ws_rows, ws_wt, bufs['save_h'], bufs['save_w'], bufs['err'])
    kernels.bpr_bwd(dt['dims'], dt['E_user'], dt['E_item'], dt['Feat'], dt['W'], dt['X'], dt['si'], dt['Y'], rng,
                    case.loss, bufs['pred'], bufs['save_h'], bufs['save_w'], bufs['loss'], bufs['gW'], bufs['gb'],
                    bufs['gu'], bufs['gi'], bufs['ku'], bufs['ki'])
    return _host(bufs, ('pred', 'save_h', 'save_w', 'gW', 'gb', 'gu', 'gi', 'ku', 'ki'))


def check_against_reference(case, pb, out, noise, mask, path):
    """Reference on the path's own row splits; asserts every output within its bound and few kink elements."""
    N = n_rows_of(case)
    if path == 'simt':
        splits = split_rows(N, *simt_geometry(N))
    else:
        _, ns, rps = bwd_geometry(N, case.F)
        splits = split_rows(N, ns, rps)
    # the fused step divides the MSE by mse_pairs; the two pairs of calls by the pairs of the call
    mse = (case.mse_pairs or case.P) if path == 'fused' else case.P
    ref = reference(pb, noise, mask, mse, splits, save_h=out['save_h'])
    fails, observed = compare(out, ref)
    n_kink = int(ref['kink'].sum())
    print('%-16s %-5s kinks %d / %d  observed C: %s' % (case.name, path, n_kink, ref['kink'].size,
          ' '.join('%s %.3g' % kv for kv in observed.items())))
    assert not fails, '%s (%s):\n  ' % (case.name, path) + '\n  '.join(fails)
    assert n_kink <= 1 + 1e-4 * ref['kink'].size, '%s: %d pre-activations within their bound of zero' % (case.name,
                                                                                                         n_kink)
    return ref


RUNNERS = {'fused': run_fused, 'tc': run_tc_pair, 'simt': run_simt}
PATH_CASES = [(c.name, p) for c in CASES for p in c.paths]


def _assert_geometry(case):
    from dccf_b200 import kernels
    N = n_rows_of(case)
    assert kernels.train_fwd_ksplits(N, case.F) == case.ks
    assert kernels.train_bwd_splits(N, case.F) == case.splits
    assert kernels.train_fused_supported(case.S, case.A, case.loss) == case.fused


@pytest.mark.parametrize('name,path', PATH_CASES)
def test_training_step_equals_float64_reference(name, path):
    import torch
    case = CASE[name]
    _assert_geometry(case)
    dev = torch.device('cuda:0')
    pb = make_problem(case)
    dt = _device_problem(pb, dev)
    rng, noise, mask = _rng(case, pb, dt, dev)
    out = RUNNERS[path](case, dt, rng, dev)
    check_against_reference(case, pb, out, noise, mask, path)


@pytest.mark.parametrize('name', ['default', 'ks5_s40a2'])
def test_fused_step_bitwise_invariants(name):
    """Outputs that must not change by one bit: the step as one call (phases 7), as three calls (1, 2, 4) and with the
    middle and dW kernels as programmatic dependents (7|16|32); all of it as 63 on W operand images prepared by
    dccf_train_prep_w_image; the middle kernel on the exposure softmax of dccf_adam_link_ids; the RNG offset read from
    device memory."""
    import torch
    case = CASE[name]
    dev = torch.device('cuda:0')
    pb = make_problem(case)
    dt = _device_problem(pb, dev)
    rng, noise, mask = _rng(case, pb, dt, dev)
    base = run_fused(case, dt, rng, dev)
    check_against_reference(case, pb, base, noise, mask, 'fused')
    variants = {'1,2,4': dict(calls=((1, False), (2, False), (4, False))),
                '7|16|32': dict(calls=((7 | 16 | 32, False),)),
                '63 on a prepared W image': dict(calls=((63, True),)),
                'expo_e / expo_den': dict(expo_split=True)}
    for label, kw in variants.items():
        got = run_fused(case, dt, rng, dev, **kw)
        for k in base:
            assert np.array_equal(np.asarray(got[k]), np.asarray(base[k])), (label, k)
    rng_dev, _, _ = _rng(case, pb, dt, dev, offset_dev=True)
    got = run_fused(case, dt, rng_dev, dev)
    for k in base:
        assert np.array_equal(np.asarray(got[k]), np.asarray(base[k])), ('offset_dev', k)


def test_fused_step_on_a_second_device_after_the_first():
    """A fused step whose middle kernel needs more than 48 KB of shared memory (S=40, A=2) on cuda:0 and then on
    cuda:1 in the same process: the shared-memory opt-in is made per device, both match the reference and the second
    device's outputs are bit-identical to the first's."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    case = CASE['ks5_s40a2']
    assert mid_smem_bytes(case.S, case.A, case.loss) > 48 * 1024
    pb = make_problem(case)
    outs = []
    for d in (0, 1):
        dev = torch.device('cuda', d)
        with torch.cuda.device(dev):
            dt = _device_problem(pb, dev)
            rng, noise, mask = _rng(case, pb, dt, dev)
            out = run_fused(case, dt, rng, dev)
        check_against_reference(case, pb, out, noise, mask, 'fused')
        outs.append(out)
    for k in outs[0]:
        assert np.array_equal(np.asarray(outs[0][k]), np.asarray(outs[1][k])), k
