"""Lock-step host emulation of kernels written after round 1's GPU budget was spent (no GPU needed).

k_gather_scores (dccf_b200/csrc/gather_scores.cu) is transcribed line by line for one warp of 32 lanes — shuffles become
index permutations of 32-element arrays — and compared with the oracle for slot counts that exercise every branch of its
schedule: Z = 1 (no confounders), 11 (default), 16 / 17 (chunk boundary), 41 (three chunks, padded last group), an odd
number of pairs (idle half-warp) and a fully idle warp.  This checks the ALGORITHM (index arithmetic, chunked max-shifted
softmax, padded slots); the CUDA code itself is checked on hardware by tests/test_gpu_zz_gather.py."""
import numpy as np
import pytest

from oracle import dccf_oracle as O

D = 64
def shfl_idx(v, src):            # v[32], src[32] -> v[src]
    return v[src]
def shfl_xor(v, o):
    return v[np.arange(32) ^ o]
def half_sum(v):
    for o in (8, 4, 2, 1): v = v + shfl_xor(v, o)
    return v
def half_max(v):
    for o in (8, 4, 2, 1): v = np.maximum(v, shfl_xor(v, o))
    return v
def expo_of(params, u, it):
    """backdoor.cuh::expo_value: the dense matrix, or the IPSBiasedMF formula on the fly (mode 1)"""
    fac = params.get('ipsmf')
    if fac is None:
        return params['expo'][u, it]
    pred = np.float32(np.dot(fac['mf_user'][u], fac['mf_item'][it])) + fac['mf_user_bias'][u] + fac['mf_item_bias'][it] \
        + fac['mf_global_bias']
    return np.float32(pred / max(fac['propensity'][it], fac['mf_min_propensity']))


def warp(params, PI, PF, X, si, n_pairs, warp_index, out):
    lane = np.arange(32); sub = lane & 15; half_base = lane & 16
    p_raw = warp_index * 2 + (lane >> 4)
    active = p_raw < n_pairs
    p = np.where(active, p_raw, n_pairs - 1)
    S = si.shape[1]; Z = S + 1
    u = X[p, 0]; fi = X[p, 1]
    cols = (4 * sub)[:, None] + np.arange(4)[None, :]
    eu = params['E_user'][u[:, None], cols]          # [32,4]
    pf = PF[fi[:, None], cols]
    run_max = np.full(32, -np.inf, np.float32); num = np.zeros(32, np.float32); den = np.zeros(32, np.float32)
    for z0 in range(0, Z, 16):
        z_mine = z0 + sub
        it_mine = fi.copy(); x_mine = np.full(32, -np.inf, np.float32)
        for l in range(32):
            if z_mine[l] < Z:
                if z_mine[l] > 0: it_mine[l] = si[p[l], z_mine[l] - 1]
                x_mine[l] = expo_of(params, u[l], it_mine[l])
        nz = min(16, Z - z0)
        s_mine = np.zeros(32, np.float32)
        for j0 in range(0, nz, 4):
            a = []
            for q in range(4):
                src = (j0 + q) if (j0 + q < nz) else 0
                it = shfl_idx(it_mine, half_base | src)
                a.append(PI[it[:, None], cols])
            for q in range(4):
                d = (np.maximum(a[q] + pf, 0) * eu).sum(1).astype(np.float32)
                d = half_sum(d)
                s_mine = np.where(sub == j0 + q, d, s_mine)
        new_max = np.maximum(run_max, half_max(x_mine))
        rescale = np.where(run_max == -np.inf, 0.0, np.exp(run_max - new_max)).astype(np.float32)
        e = np.where(z_mine < Z, np.exp(x_mine - new_max), 0.0).astype(np.float32)
        num = num * rescale + half_sum(e * s_mine)
        den = den * rescale + half_sum(e)
        run_max = new_max
    for l in range(32):
        if active[l] and sub[l] == 0: out[p_raw[l]] = num[l] / den[l]


def _problem(seed, U, I, F, P, S):
    rs = np.random.RandomState(seed)
    params = {'E_user': (rs.standard_normal((U, 64)) * 0.05).astype(np.float32),
              'E_item': (rs.standard_normal((I, 64)) * 0.05).astype(np.float32),
              'W': (rs.standard_normal((64, 64 + F)) * 0.05).astype(np.float32),
              'b': (rs.standard_normal(64) * 0.05).astype(np.float32),
              'Feat': (rs.standard_normal((I, F)) / np.sqrt(F)).astype(np.float32),
              'expo': rs.random_sample((U, I)).astype(np.float32)}
    X = np.stack([rs.randint(0, U, P), rs.randint(0, I, P)], 1).astype(np.int64)
    si = rs.randint(0, I, size=(P, S)).astype(np.int64)
    return params, X, si


@pytest.mark.parametrize('P,S,A,ipsmf', [(7, 10, 2, False), (5, 40, 1, False), (3, 0, 2, False), (4, 15, 1, False),
                                        (6, 16, 3, False), (1, 10, 2, False), (9, 10, 2, True)])
def test_gather_scorer_schedule_emulated(P, S, A, ipsmf):
    U, I, F = 30, 50, 64
    params, X, si = _problem(21 + S, U, I, F, P, S)
    fac = None
    if ipsmf:
        from dccf_b200 import synth
        fac = synth.make_ipsmf_factors(U, I, seed=3)
        params['ipsmf'] = fac
    W = params['W'].astype(np.float64)
    PI = (params['E_item'].astype(np.float64) @ W[:, :64].T).astype(np.float32)              # dccf_tc_prepare's tables
    PF = (params['Feat'].astype(np.float64) @ W[:, 64:].T + params['b']).astype(np.float32)
    out = np.full(P, np.nan, np.float32)
    with np.errstate(invalid='ignore'):
        for w in range((P + 1) // 2 + 1):                # + one fully idle warp
            warp(params, PI, PF, X, si, P, w, out)
    ref = O.predict(params, X, si, None, None, A, dtype=np.float64, expo=fac)['pred']
    assert np.isfinite(out).all()
    assert np.abs(out - ref).max() / np.abs(ref).max() < 1e-5


# ---------------------------------------------------------------------------------------------------------
# Index arithmetic of two optimizer kernels whose launch shapes changed late in round 2 (adam.cu)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n_rec', [(1, 1), (256, 2816), (2048, 22528), (300, 0), (257, 513)])
def test_csr_build_ctas_visit_every_record_once(n_rec):
    """k_csr_build: the tables' record ranges are laid out in blocks of 256 records (link_lo / link_n, marshal_adam);
    dccf_adam_csr_build launches one 256-thread CTA per block.  Transcription of the kernel's mapping blockIdx.x,
    threadIdx.x -> (table, record): every record of every table exactly once, nothing else."""
    tables, lo = [], 0
    for n in n_rec:                                   # marshal_adam: link_n = ceil(n_rec / 256) blocks per table
        link_n = (n + 255) // 256
        tables.append({'n_rec': n, 'link_lo': lo, 'link_n': link_n})
        lo += link_n
    link_blocks = lo
    seen = [np.zeros(t['n_rec'], dtype=np.int64) for t in tables]
    for block in range(link_blocks):
        for i, t in enumerate(tables):
            b = block - t['link_lo']
            if b < 0 or b >= t['link_n']:
                continue
            r = b * 256 + np.arange(256)
            r = r[r < t['n_rec']]
            seen[i][r] += 1
            break                                     # (the kernel returns after the table that owns the block)
    for s in seen:
        assert (s == 1).all()


@pytest.mark.parametrize('n_rows,block_n,cta_threads', [(64000, 148, 224), (48000, 111, 224), (16000, 37, 224), (5, 3, 128),
                                                        (4 * 7 * 3 + 1, 3, 224), (1025, 148, 256)])
def test_untouched_sweep_pipeline_covers_every_row_once(n_rows, block_n, cta_threads):
    """k_adam_untouched: a warp owns rows 4w .. 4w+3 per trip (two per half-warp); the touched flags of the NEXT trip are
    read, and its rows requested into L2, one trip ahead.  Transcription of the loop: every untouched row is updated
    exactly once, no touched row is, and the flags consumed in a trip are the ones loaded for exactly those rows."""
    rng = np.random.default_rng(n_rows)
    head = np.where(rng.random(n_rows) < 0.05, 3, -1)                 # -1 = untouched
    updated = np.zeros(n_rows, dtype=np.int64)
    n_warps = (block_n * cta_threads) >> 5

    def row_ok(r):
        return r < n_rows and head[r] == -1

    for warp in range(n_warps):
        for half in (0, 1):
            v0 = 4 * warp < n_rows and row_ok(4 * warp + half)
            v1 = 4 * warp < n_rows and row_ok(4 * warp + half + 2)
            w = warp
            while 4 * w < n_rows:
                r0, r1 = 4 * w + half, 4 * w + half + 2
                n0, n1 = r0 + 4 * n_warps, r0 + 4 * n_warps + 2
                nv0, nv1 = row_ok(n0), row_ok(n1)                     # loaded before this trip's rows
                assert v0 == row_ok(r0) and v1 == row_ok(r1)          # the flags in hand belong to this trip's rows
                if v0:
                    updated[r0] += 1
                if v1:
                    updated[r1] += 1
                v0, v1 = nv0, nv1
                w += n_warps
    assert (updated[head == -1] == 1).all() and (updated[head != -1] == 0).all()
