"""The BiasedMF / IPSBiasedMF kernels (csrc/mf.cu) against a float64 reference, element by element, over their launch
geometry.

The reference (tests/mf_reference.py: `pairs` per pair, `gradients` per row) is fed the exact float32 values the
kernels read.  Each element is bounded by

    |y_kernel - y_ref| <= C * 2^-20 * |y|_abs + 2 ulp(y_ref) + 2^-120

where |y|_abs carries every input's magnitude through the computation to first order (the `A_*` of `pairs`, plus the
rounding of every sum the kernel forms: n - 1 times the sum of |terms| for a sum of n terms).  The absolute 2^-120
covers the BPR sigmoid past x = 88.7, where float32 expf overflows and the true value is below 2^-127 / M.  C is per
output, about 4 times the largest value a B200 needed; each test prints what it needed ("observed C").

What has an exact answer is compared bit for bit: the record keys, each CTA's global-bias partial (the float32 sum of
its own bias records in half-warp order, dead half-warps counting 0), the bias gradients of k_mf_bias_grad (the float32
sum of a row's records in ascending record index, exactly 0 for untouched rows) and its loss (the partials summed in
index order, times loss_scale).

  a. k_mf_step through kernels.mf_step, at batch sizes that leave partial last CTAs and hand a BPR pair's negative to
     a CTA other than the one its index falls in, with propensities at and around the clamp M, BPR margins past
     expf's overflow and MSE errors of exactly 0.
  b. k_mf_bias_grad after the real dccf_adam_link_ids + dccf_adam_csr_build, with rows of 0 to 1024 records and
     U + I on both sides of the 256-thread block.
  c. k_mf_scores, with global_bias read from device memory.
  d. BiasedMF / IPSBiasedMF.train_step (eager, graph replays, a device-resident epoch and a ragged tail) against the
     float64 step recomputed from a snapshot of the parameters and the optimizer state, with every term visible and a
     clip that acts.

The kernel each case runs is read from a torch.profiler trace of the call.  test_mf_reference_cpu.py pins the geometry
mirror below to the library, checks that each case reaches what it claims and runs negative controls on the
comparators."""
import collections

import numpy as np
import pytest
import torch

from mf_reference import pairs

D = 64
UNIT = 2.0 ** -20
ULPS = 2
TINY = 2.0 ** -120
# about 4 times the largest C each output needed over this module on an NVIDIA B200 at a 1000 W power limit (the tests
# print "observed C"): k_mf_step pred 0.031, gb_rec 0.029, gu_rec 0.033, gi_rec 0.033, loss_part 0.0089; k_mf_scores
# 0.149; the model's step p 0.034, m 0.036, v 0.037, s 0.044, pred 0.036.  The model's loss never needed more than its
# ulps; its C is nominal.
C = {'pred': 0.12, 'gb_rec': 0.12, 'gu_rec': 0.13, 'gi_rec': 0.13, 'loss_part': 0.04, 'scores': 0.6}
C_MODEL = {'p': 0.14, 'm': 0.15, 'v': 0.15, 's': 0.18, 'pred': 0.15, 'loss': 0.05}
M_IPS = float(np.float32(0.1))
PAIRS_PER_CTA = 16
ALL = ('adam', 'gd', 'adagrad')


# ------------------------------------------------------------------------------------------------------------------
# launch geometry of k_mf_step (Python mirror, pinned to dccf_mf_step_ctas in test_mf_reference_cpu.py)
# ------------------------------------------------------------------------------------------------------------------
def step_ctas(P):
    return 0 if P <= 0 else -(-P // PAIRS_PER_CTA)


def pair_slots(P, rank):
    """(CTA, half-warp) of every pair.  Half-warp k of a CTA is threads 16k .. 16k + 15, so warp w of the grid is
    half-warps 2 (w % 8) and 2 (w % 8) + 1 of CTA w // 8.  BPR: warp w holds pair w (half 0) and its negative w + P/2
    (half 1); MSE: pairs 2w and 2w + 1."""
    p = np.arange(P)
    if rank == 1:
        b = P // 2
        w, half = np.where(p < b, p, p - b), (p >= b).astype(np.int64)
    else:
        w, half = p // 2, p % 2
    return w // 8, 2 * (w % 8) + half


# ------------------------------------------------------------------------------------------------------------------
# problems: parameters with propensity edges, BPR margins from 0 to 300 and an exactly representable prediction
# ------------------------------------------------------------------------------------------------------------------
EDGE_ITEMS = 5                    # items 0..4: propensity 0, M / 2, M, the float after M, 1
MARGINS = (0.25, 2.5, 11.0, 22.0, 43.9, 44.5, 60.0, 150.0)     # items 5 + 2k (+B) and 6 + 2k (-B), propensity 1
EXACT_ITEM = EDGE_ITEMS + 2 * len(MARGINS)      # with user 0: pred = (0 + 0.5 + 0.25 + 0.125) / 1 = 0.875 exactly
EXACT_PRED = 0.875


def make_params(rs, U, I, cls):
    """float32 parameters, propensity and M.  cls 'ips': random propensity with the edge items; 'biased': BiasedMF's
    all-ones propensity with M = 1."""
    prm = {'E_user': (rs.standard_normal((U, D)) * 0.15).astype(np.float32),
           'E_item': (rs.standard_normal((I, D)) * 0.15).astype(np.float32),
           'user_bias': (rs.standard_normal(U) * 0.3).astype(np.float32),
           'item_bias': (rs.standard_normal(I) * 0.3).astype(np.float32),
           'global_bias': np.float32(0.125)}
    if cls == 'ips':
        prop, M = rs.random_sample(I).astype(np.float32), M_IPS
        prop[:EDGE_ITEMS] = [0.0, M / 2, M, np.nextafter(np.float32(M), np.float32(2)), 1.0]
    else:
        prop, M = np.ones(I, np.float32), 1.0
    for k, B in enumerate(MARGINS):
        prm['item_bias'][EDGE_ITEMS + 2 * k], prm['item_bias'][EDGE_ITEMS + 2 * k + 1] = B, -B
        prop[EDGE_ITEMS + 2 * k:EDGE_ITEMS + 2 * k + 2] = 1.0
    prm['E_user'][0] = 0.0
    prm['user_bias'][0] = 0.5
    prm['item_bias'][EXACT_ITEM], prop[EXACT_ITEM] = 0.25, 1.0
    return prm, prop, M


def make_batch(rs, U, I, P, rank):
    """X [P, 2] int64 and Y [P] float32 that cycle through the edge values: BPR pairs with x = 0 exactly (negative =
    positive), margins +-2B, edge-propensity items and the exact prediction; MSE pairs with e = 0 exactly, edge items and
    the margin items."""
    X = np.stack([rs.randint(1, U, P), rs.randint(EXACT_ITEM + 1, I, P)], 1).astype(np.int64)
    Y = rs.randint(1, 6, P).astype(np.float32)
    if rank == 1:
        b = P // 2
        for j in range(b):
            k, m = (j + b) % 6, (j // 6) % len(MARGINS)
            if k == 0:
                X[b + j, 1] = X[j, 1]
            elif k in (1, 2):
                X[j, 1], X[b + j, 1] = EDGE_ITEMS + 2 * m + (k == 2), EDGE_ITEMS + 2 * m + (k == 1)
            elif k == 3:
                X[j, 1], X[b + j, 1] = (j // 6) % EDGE_ITEMS, (j // 6 + 1) % EDGE_ITEMS
            elif k == 4:
                X[j, 0], X[j, 1] = 0, EXACT_ITEM
        X[b:, 0] = X[:b, 0]
        Y = np.r_[np.ones(b), np.zeros(P - b)].astype(np.float32)
    else:
        for p in range(P):
            k = (p + 1) % 5
            if k == 0:
                X[p] = (0, EXACT_ITEM)
                Y[p] = EXACT_PRED
            elif k == 1:
                X[p, 1] = (p // 5) % EDGE_ITEMS
            elif k == 2:
                X[p, 1] = EDGE_ITEMS + (p // 5) % (2 * len(MARGINS))
    return X, Y


def params64(prm):
    return {k: np.asarray(v, np.float64) for k, v in prm.items()}


SCase = collections.namedtuple('SCase', 'name rank P U I cls')
BPR_P = (2, 14, 16, 18, 30, 32, 34, 254, 256, 258, 1026)
MSE_P = (1, 15, 16, 17, 31, 33, 255, 257)
STEP_CASES = ([SCase('bpr_%d' % P, 1, P, 40, 90, 'ips') for P in BPR_P] +
              [SCase('mse_%d' % P, 0, P, 40, 90, 'ips') for P in MSE_P] +
              [SCase('bpr_256_biased', 1, 256, 40, 90, 'biased'), SCase('mse_255_biased', 0, 255, 40, 90, 'biased')])
PAD = 48                          # pairs of padding after every per-pair buffer (a whole CTA and more)


def make_step_problem(c, seed=0):
    rs = np.random.RandomState(1000 + seed)
    prm, prop, M = make_params(rs, c.U, c.I, c.cls)
    X, Y = make_batch(rs, c.U, c.I, c.P, c.rank)
    return dict(case=c, prm=prm, prop=prop, M=M, X=X, Y=Y,
                ref=pairs(params64(prm), X, Y, c.rank, prop.astype(np.float64), M))


# ------------------------------------------------------------------------------------------------------------------
# comparators
# ------------------------------------------------------------------------------------------------------------------
def ulp(x):
    return np.spacing(np.abs(np.asarray(x, np.float32))).astype(np.float64)


def judge(got, ref, A, c):
    """(failing elements, the C each element needs)."""
    got = np.asarray(got, np.float64)
    slack = ULPS * ulp(ref) + TINY
    with np.errstate(invalid='ignore', over='ignore', divide='ignore'):
        d = np.abs(got - ref)
        bad = ~(d <= c * UNIT * A + slack)
        need = np.where(d <= slack, 0.0, (d - slack) / (UNIT * A))
    return bad, np.nan_to_num(need, nan=np.inf)


def g_part_of(gb_rec, P, rank, drop_last=False):
    """The global-bias partial of every CTA: float32 sum, in half-warp order, of its bias records (dead half-warps 0)."""
    n = step_ctas(P)
    cta, hw = pair_slots(P, rank)
    s = np.zeros((n, PAIRS_PER_CTA), np.float32)
    s[cta, hw] = gb_rec[:P]
    acc = np.zeros(n, np.float32)
    for k in range(PAIRS_PER_CTA - (1 if drop_last else 0)):
        acc = (acc + s[:, k]).astype(np.float32)
    return acc


def loss_part_ref(pb):
    """float64 loss terms of every CTA and their magnitude (16 terms summed in float32)."""
    c, ref = pb['case'], pb['ref']
    n = step_ctas(c.P)
    cta, _ = pair_slots(c.P, c.rank)
    lp, A, ab = np.zeros(n), np.zeros(n), np.zeros(n)
    np.add.at(lp, cta, ref['term'])
    np.add.at(A, cta, ref['A_term'])
    np.add.at(ab, cta, np.abs(ref['term']))
    return lp, A + (PAIRS_PER_CTA - 1) * ab + np.abs(lp)


def check_step(pb, out, observed, cs=None):
    """{output: failing elements} of one k_mf_step call; records the C each output needed."""
    cs = C if cs is None else cs
    c, ref, X = pb['case'], pb['ref'], pb['X']
    P, n = c.P, step_ctas(c.P)
    fails = {}

    def elementwise(name, got, want, A):
        bad, need = judge(got, want, A, cs[name])
        fails[name] = int(bad.sum())
        observed[name] = max(observed.get(name, 0.0), float(need.max()) if need.size else 0.0)

    elementwise('pred', out['pred'][:P], ref['pred'], ref['A_pred'])
    elementwise('gb_rec', out['gb_rec'][:P], ref['r'], ref['A_r'])
    elementwise('gu_rec', out['gu_rec'][:P], ref['gu'], ref['A_gu'])
    elementwise('gi_rec', out['gi_rec'][:P], ref['gi'], ref['A_gi'])
    lp, A_lp = loss_part_ref(pb)
    elementwise('loss_part', out['loss_part'][:n], lp, A_lp)
    fails['keys'] = int((out['keys_u'][:P] != X[:, 0]).sum() + (out['keys_i'][:P] != X[:, 1]).sum())
    fails['g_part'] = int((out['g_part'][:n].view(np.int32) != g_part_of(out['gb_rec'], P, c.rank).view(np.int32)).sum())
    # nothing is written past the batch or past the last CTA (the buffers come back with their sentinels)
    fails['past the end'] = int(sum((~np.isnan(out[k][P:])).sum() for k in ('pred', 'gb_rec', 'gu_rec', 'gi_rec')) +
                                (out['keys_u'][P:] != -7).sum() + (out['keys_i'][P:] != -7).sum() +
                                (~np.isnan(out['g_part'][n:])).sum() + (~np.isnan(out['loss_part'][n:])).sum())
    return fails


def row_sums_f32(keys, gb_rec, n_rows, order='ascending', drop_first=False):
    """float32 sum of each row's records in ascending record index (0 for untouched rows)."""
    out = np.zeros(n_rows, np.float32)
    for row in np.unique(keys):
        idx = np.flatnonzero(keys == row)
        if order == 'descending':
            idx = idx[::-1]
        if drop_first and len(idx) > 1:
            idx = idx[1:]
        acc = gb_rec[idx[0]]
        for j in idx[1:]:
            acc = np.float32(acc + gb_rec[j])
        out[row] = acc
    return out


def loss_of(loss_part, loss_scale):
    acc = np.float32(0.0)
    for x in loss_part:
        acc = np.float32(acc + x)
    return np.float32(acc * np.float32(loss_scale))


def check_bias(pb, out):
    """{output: elements that differ bit for bit} of one k_mf_bias_grad call."""
    X, gb = pb['X'], pb['gb_rec']
    fails = {}
    for name, col, n in (('g_user', 0, pb['U']), ('g_item', 1, pb['I'])):
        want = row_sums_f32(X[:, col].astype(np.int32), gb, n)
        fails[name] = int((out[name][:n].view(np.int32) != want.view(np.int32)).sum())
        fails[name + ' past the end'] = int((~np.isnan(out[name][n:])).sum())
    want = loss_of(pb['loss_part'], pb['loss_scale'])
    fails['loss'] = int(out['loss'][:1].view(np.int32)[0] != np.asarray(want).view(np.int32))
    return fails


def _report(observed, name):
    print('observed C %s: %s' % (name, ', '.join('%s %.3g' % kv for kv in sorted(observed.items()))))


# ------------------------------------------------------------------------------------------------------------------
# b. bias gradient problems: planted record counts, U + I around the 256-thread block, hot rows
# ------------------------------------------------------------------------------------------------------------------
BCase = collections.namedtuple('BCase', 'name U I P hot')
COUNTS = (1, 2, 3, 17)
BIAS_CASES = [BCase('u+i_100', 40, 60, 96, None), BCase('u+i_255', 100, 155, 130, None),
              BCase('u+i_256', 128, 128, 200, None), BCase('u+i_257', 57, 200, 160, None),
              BCase('blocks', 700, 1500, 1024, None), BCase('one_item', 300, 500, 1024, 'item'),
              BCase('one_user', 300, 500, 1024, 'user')]


def _planted(rs, n_rows, P):
    """P keys with one row per count of COUNTS, the rest over half of the remaining rows (the others untouched)."""
    rows = rs.permutation(n_rows)
    planted, rest = rows[:len(COUNTS)], rows[len(COUNTS):len(COUNTS) + max(1, (n_rows - len(COUNTS)) // 2)]
    keys = np.concatenate([np.full(k, r) for r, k in zip(planted, COUNTS)] + [rs.choice(rest, P - sum(COUNTS))])
    return keys[rs.permutation(P)]


def make_bias_problem(c, seed=0):
    rs = np.random.RandomState(2000 + seed)
    X = np.stack([_planted(rs, c.U, c.P), _planted(rs, c.I, c.P)], 1).astype(np.int64)
    if c.hot == 'item':
        X[:, 1] = c.I // 3
    elif c.hot == 'user':
        X[:, 0] = c.U // 3
    # records and loss partials over 40 binades: every summation order gives a different float32 result
    gb = (rs.standard_normal(c.P) * 2.0 ** rs.randint(-20, 20, c.P)).astype(np.float32)
    n = step_ctas(c.P)
    lp = (rs.random_sample(n) * 2.0 ** rs.randint(-12, 12, n)).astype(np.float32)
    return dict(case=c, U=c.U, I=c.I, X=X, gb_rec=gb, loss_part=lp, loss_scale=1.0 / c.P if seed % 2 else 1.0)


# ------------------------------------------------------------------------------------------------------------------
# device runs
# ------------------------------------------------------------------------------------------------------------------
def traced(fn):
    """(fn(), names of the CUDA kernels it launched, spaces removed), from a torch.profiler trace.  A torch kernel runs
    first in the same trace: after other modules' profiler sessions and graph captures in one process, a trace holding
    only the library's launches has come back without kernel records, one that also holds a torch launch has not."""
    from torch.profiler import ProfilerActivity, profile
    probe = torch.zeros(1, device='cuda')
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        probe.add_(1)
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name.replace(' ', '') for e in prof.events()}


def launched(names, kernel):
    return any('dccf::%s(' % kernel in n for n in names)


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _padded_ids(X, U, I):
    """X on the device with PAD rows of valid ids after it (a kernel reading past the batch reads ids, not garbage)."""
    full = np.concatenate([X, np.stack([np.arange(PAD) % U, np.arange(PAD) % I], 1)]).astype(np.int64)
    return _cuda(full)


def run_step(pb):
    from dccf_b200 import kernels
    c, prm = pb['case'], pb['prm']
    P, n = c.P, step_ctas(c.P)
    X = _padded_ids(pb['X'], c.U, c.I)
    Y = _cuda(np.r_[pb['Y'], np.zeros(PAD, np.float32)])
    nan = lambda *s: torch.full(s, float('nan'), dtype=torch.float32, device='cuda')      # noqa: E731
    out = {'pred': nan(P + PAD), 'gb_rec': nan(P + PAD), 'gu_rec': nan(P + PAD, D), 'gi_rec': nan(P + PAD, D),
           'keys_u': torch.full((P + PAD,), -7, dtype=torch.int32, device='cuda'),
           'keys_i': torch.full((P + PAD,), -7, dtype=torch.int32, device='cuda'),
           'g_part': nan(n + 4), 'loss_part': nan(n + 4)}
    err = torch.zeros(1, dtype=torch.int32, device='cuda')
    dev = {k: _cuda(np.asarray(v, np.float32).reshape(-1) if k == 'global_bias' else v) for k, v in prm.items()}

    def call():
        kernels.mf_step(dev['E_user'], dev['E_item'], dev['user_bias'], dev['item_bias'], dev['global_bias'],
                        _cuda(pb['prop']), pb['M'], X[:P], Y[:P] if c.rank == 0 else None, 1 - c.rank, out['pred'],
                        out['gu_rec'], out['gi_rec'], out['gb_rec'], out['keys_u'], out['keys_i'], out['g_part'],
                        out['loss_part'], err)
    _, names = traced(call)
    assert launched(names, 'k_mf_step'), names
    assert int(err) == 0
    return {k: v.cpu().numpy() for k, v in out.items()}


def run_bias(pb):
    from dccf_b200 import kernels
    c = pb['case']
    U, I, P = c.U, c.I, c.P
    i32 = lambda n, v=0: torch.full((n,), v, dtype=torch.int32, device='cuda')      # noqa: E731
    X = _cuda(pb['X'])
    tabs = []
    for n_rows in (U, I):
        t = dict(p=torch.zeros((n_rows, D), device='cuda'), keys=i32(P), grads=torch.zeros((P, D), device='cuda'),
                 head=i32(n_rows, -1), next=i32(P, 7), csr=(i32(P, -5), i32(n_rows, -5), i32(2 * P, -5), i32(2)))
        tabs.append(t)
    tables = [kernels.adam_table(t['p'], None, None, t['keys'], t['grads'], 1, P, P, P * D, t['head'], t['next'],
                                 csr=t['csr']) for t in tabs]
    kernels.adam_link_ids(kernels.make_dims(U, I, 0, 0, 1), X, None, tabs[0]['head'], tabs[0]['next'], tabs[1]['head'],
                          tabs[1]['next'], n_seg=1,
                          extra=kernels.make_link_extra(rec_rows=(tabs[0]['csr'][0], tabs[1]['csr'][0])))
    kernels.adam_csr_build(tables)
    out = {'g_user': torch.full((U + 5,), float('nan'), device='cuda'),
           'g_item': torch.full((I + 5,), float('nan'), device='cuda'),
           'loss': torch.full((2,), float('nan'), device='cuda')}
    gb, lp = _cuda(pb['gb_rec']), _cuda(pb['loss_part'])
    _, names = traced(lambda: kernels.mf_bias_grad(tables[0], tables[1], gb, out['g_user'], out['g_item'], lp, len(lp),
                                                   pb['loss_scale'], out['loss']))
    assert launched(names, 'k_mf_bias_grad'), names
    return {k: v.cpu().numpy() for k, v in out.items()}


pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------------------
# a. k_mf_step
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('case', STEP_CASES, ids=[c.name for c in STEP_CASES])
def test_mf_step_against_float64_reference(case):
    pb = make_step_problem(case, STEP_CASES.index(case))
    observed = {}
    fails = check_step(pb, run_step(pb), observed)
    _report(observed, case.name)
    assert not any(fails.values()), fails


# ------------------------------------------------------------------------------------------------------------------
# b. k_mf_bias_grad
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('case', BIAS_CASES, ids=[c.name for c in BIAS_CASES])
def test_mf_bias_grad_is_the_ascending_float32_sum(case):
    for seed in (0, 1):
        pb = make_bias_problem(case, seed)
        fails = check_bias(pb, run_bias(pb))
        assert not any(fails.values()), (seed, fails)


# ------------------------------------------------------------------------------------------------------------------
# c. k_mf_scores
# ------------------------------------------------------------------------------------------------------------------
SCORE_N = (1, 255, 256, 257, 65537)


@pytest.mark.parametrize('cls', ['ips', 'biased'])
@pytest.mark.parametrize('n', SCORE_N)
def test_mf_scores_against_float64_reference(n, cls):
    """Element by element at n pairs, with the edge propensities; then global_bias changed on the device between two
    calls with the same factors: the second call must use the new value."""
    from dccf_b200 import kernels
    from mf_reference import forward
    rs = np.random.RandomState(n)
    U, I = 300, 400
    prm, prop, M = make_params(rs, U, I, cls)
    X = np.stack([rs.randint(0, U, n), rs.randint(0, I, n)], 1).astype(np.int64)
    X[:min(n, 3 * EDGE_ITEMS), 1] = np.arange(min(n, 3 * EDGE_ITEMS)) % EDGE_ITEMS
    fac = {'mf_user': _cuda(prm['E_user']), 'mf_item': _cuda(prm['E_item']), 'mf_user_bias': _cuda(prm['user_bias']),
           'mf_item_bias': _cuda(prm['item_bias']), 'propensity': _cuda(prop), 'mf_min_propensity': M}
    g = torch.tensor([float(prm['global_bias'])], dtype=torch.float32, device='cuda')
    Xd = _cuda(X)
    out = torch.full((n + 7,), float('nan'), device='cuda')
    observed = {}
    for gval in (0.125, -3.75):
        g.fill_(gval)
        _, names = traced(lambda: kernels.mf_scores(fac, g, Xd, out[:n]))
        assert launched(names, 'k_mf_scores'), names
        got = out.cpu().numpy()
        p64 = dict(params64(prm), global_bias=np.float64(gval))
        pred, _, mag = forward(p64, X, prop.astype(np.float64), M)
        bad, need = judge(got[:n], pred, mag + np.abs(pred), C['scores'])
        observed['scores'] = max(observed.get('scores', 0.0), float(need.max()))
        assert not bad.any(), (gval, int(bad.sum()))
        assert np.isnan(got[n:]).all()
    _report(observed, 'scores n=%d %s' % (n, cls))


# ------------------------------------------------------------------------------------------------------------------
# d. the model's step
# ------------------------------------------------------------------------------------------------------------------
def model_batch(rs, U, I, P, rank):
    """A batch over the first half of each table (the rest stays untouched) with a hot user and a hot item."""
    X = np.stack([rs.randint(0, U // 2, P), rs.randint(0, I // 2, P)], 1).astype(np.int64)
    X[:17, 1] = 5
    if rank == 1:
        X[:8, 0] = 3
        X[P // 2:, 0] = X[:P // 2, 0]
        Y = np.r_[np.ones(P // 2), np.zeros(P - P // 2)].astype(np.float32)
    else:
        X[-17:, 0] = 3
        Y = rs.randint(1, 6, P).astype(np.float32)
    return X, Y


def _snapshot(model):
    opt = model.optimizer
    names = {'adam': ('m', 'v'), 'gd': (), 'adagrad': ('s',)}[opt.kind]
    params = {k: p.data.detach().cpu().numpy().copy() for k, p in opt.params.items()}
    st = {k: dict(zip(names, [x.cpu().numpy().copy() for x in opt.state_of(k) if x is not None])) for k in opt.params}
    return params, st, opt.step_count


def step_gradients(p0, X, Y, rank, prop, M):
    """float64 gradient of every parameter for the step from p0, and its magnitude with the rounding of each sum the
    kernels form (a row's records; the global bias: 16 records per CTA, then the CTA partials)."""
    f = {k: np.asarray(v, np.float64).reshape(-1) if 'bias' in k else np.asarray(v, np.float64) for k, v in p0.items()}
    pr = pairs(f, X, Y, rank, prop, M)
    u, i = X[:, 0], X[:, 1]
    gs, A = {}, {}
    for k, rows, g, a in (('E_user', u, pr['gu'], pr['A_gu']), ('E_item', i, pr['gi'], pr['A_gi']),
                          ('user_bias', u, pr['r'], pr['A_r']), ('item_bias', i, pr['r'], pr['A_r'])):
        n_rows = p0[k].shape[0]
        s, m, ab = (np.zeros((n_rows,) + g.shape[1:]) for _ in range(3))
        np.add.at(s, rows, g)
        np.add.at(m, rows, a)
        np.add.at(ab, rows, np.abs(g))
        cnt = np.bincount(rows, minlength=n_rows).reshape((n_rows,) + (1,) * (g.ndim - 1))
        gs[k], A[k] = s.reshape(p0[k].shape), (m + np.maximum(cnt - 1, 0) * ab).reshape(p0[k].shape)
    n = step_ctas(len(X))
    gs['global_bias'] = np.asarray(pr['r'].sum())
    A['global_bias'] = np.asarray(pr['A_r'].sum() + (PAIRS_PER_CTA + n) * np.abs(pr['r']).sum())
    loss = pr['term'].sum()
    A_loss = pr['A_term'].sum() + (PAIRS_PER_CTA + n) * np.abs(pr['term']).sum()
    if rank == 0:
        loss, A_loss = loss / len(X), A_loss / len(X)
    return gs, A, pr, loss, A_loss + abs(loss)


def model_step_errors(model, before, X, Y, rank, out, observed):
    """The step just taken, recomputed in float64 from the snapshot `before`."""
    from test_gpu_optimizer_reference import compare
    opt = model.optimizer
    p0, s0, t0 = before
    p1, s1, t = _snapshot(model)
    assert t == t0 + 1
    prop, M = model._scale()
    gs, A, pr, loss, A_loss = step_gradients(p0, X, Y, rank, prop.cpu().numpy().astype(np.float64), M)
    hp = dict(rule=opt.kind, lr=opt.lr, l2=opt.l2, wd=opt.weight_decay, clip=opt.clip, eps=opt.eps, beta1=opt.beta1,
              beta2=opt.beta2, t=t)
    errors = []
    for k in p0:
        fails, need = compare(opt.kind, hp, p0[k], s0[k], gs[k], A[k], dict({'p': p1[k]}, **s1[k]), cs=C_MODEL)
        for o, v in need.items():
            observed[o] = max(observed.get(o, 0.0), v)
        if fails['any']:
            errors.append((t, k, fails, need))
    for name, got, want, a in (('pred', out['prediction'], pr['pred'], pr['A_pred']),
                               ('loss', out['loss'], np.asarray(loss), np.asarray(A_loss))):
        bad, need = judge(got.detach().cpu().numpy().reshape(np.shape(want)), want, a, C_MODEL[name])
        observed[name] = max(observed.get(name, 0.0), float(np.max(need)))
        if bad.any():
            errors.append((t, name, int(bad.sum())))
    model.check_ids()
    return errors


def run_model_sequence(cls, kind, rank, clip=None, seed=0):
    """Eager first step, graph capture and replays, a device-resident epoch, then a ragged last batch; every step
    checked against the float64 step from the snapshot before it.  Returns (errors, observed C)."""
    from test_gpu_mf import make_model
    U, I, P, tail = 120, 200, 64, 40 if rank == 1 else 37
    rs = np.random.RandomState(30 + seed)
    prop = None
    if cls == 'IPSBiasedMF':
        prop = rs.random_sample(I).astype(np.float32)
        prop[:4] = [0.0, M_IPS / 2, M_IPS, 1.0]
    model = make_model(U, I, seed=7 + seed, prop=prop, M=M_IPS, scale=10.0, cls=cls)
    hp = {'lr': 0.05, 'l2': 1e-3}
    batches = [model_batch(rs, U, I, P, rank) for _ in range(8)] + [model_batch(rs, U, I, tail, rank)]
    kw = {}
    if clip == 'median':
        # the clip at about the median |g| of the first step's touched elements, so that it acts on half of them
        params = {'E_user': model.uid_embeddings.weight, 'E_item': model.iid_embeddings.weight,
                  'user_bias': model.user_bias.weight, 'item_bias': model.item_bias.weight,
                  'global_bias': model.global_bias}
        params = {k: v.detach().cpu().numpy() for k, v in params.items()}
        sc, M = model._scale()
        gs = step_gradients(params, batches[0][0], batches[0][1], rank, sc.cpu().numpy().astype(np.float64), M)[0]
        g1 = np.concatenate([(gs[k] + 2 * hp['l2'] * params[k])[np.abs(gs[k]) > 0] for k in ('E_user', 'E_item')])
        kw['clip'] = float(np.float32(np.median(np.abs(g1))))
    model.optimizer = model.make_fused_optimizer(lr=hp['lr'], l2=hp['l2'], kind=kind, **kw)
    model.use_cuda_graph = True
    errors, observed = [], {}

    def feed(X, Y):
        return {'X': _cuda(X), 'Y': _cuda(Y), 'rank': rank, 'train': True, 'dropout': 0.0}

    # eager first step (traced), then three replays of the captured graph
    for b in range(4):
        X, Y = batches[b]
        before = _snapshot(model)
        if b == 0:
            out, names = traced(lambda: model.train_step(feed(X, Y)))
            assert launched(names, 'k_mf_step') and launched(names, 'k_mf_bias_grad'), names
        else:
            out = model.train_step(feed(X, Y))
            torch.cuda.synchronize()
        errors += model_step_errors(model, before, X, Y, rank, out, observed)
    assert any(isinstance(v, dict) and not k[3] for k, v in model._graphs.items())        # the replays did run
    # a device-resident epoch: its first batch eager, then one launch of the staged graph per batch
    epoch = batches[4:8]
    X_ep = _cuda(np.stack([e[0] for e in epoch]))
    Y_ep = _cuda(np.stack([e[1] for e in epoch])) if rank == 0 else None
    before = _snapshot(model)
    step = model.begin_resident_epoch(X_ep, X_ep[:, :, :0], 0.0, Y_epoch=Y_ep)
    torch.cuda.synchronize()
    assert step is not None and step.remaining() == len(epoch) - 1
    errors += model_step_errors(model, before, epoch[0][0], epoch[0][1], rank, step.first, observed)
    for b in range(1, len(epoch)):
        before = _snapshot(model)
        out = step()
        torch.cuda.synchronize()
        errors += model_step_errors(model, before, epoch[b][0], epoch[b][1], rank, out, observed)
    assert any(isinstance(v, dict) and k[3] for k, v in model._graphs.items())            # the staged graph ran
    # the ragged last batch
    X, Y = batches[8]
    before = _snapshot(model)
    out = model.train_step(feed(X, Y))
    torch.cuda.synchronize()
    errors += model_step_errors(model, before, X, Y, rank, out, observed)
    assert model.optimizer.step_count == 9
    return errors, observed, kw.get('clip')


@pytest.mark.parametrize('rank', [1, 0])
@pytest.mark.parametrize('kind', ALL)
@pytest.mark.parametrize('cls', ['IPSBiasedMF', 'BiasedMF'])
def test_model_steps_against_float64_reference(cls, kind, rank):
    errors, observed, _ = run_model_sequence(cls, kind, rank)
    _report(observed, '%s %s rank %d' % (cls, kind, rank))
    assert not errors, errors[:6]


@pytest.mark.parametrize('kind,rank', [('adam', 1), ('gd', 0)])
def test_model_steps_with_an_active_clip(kind, rank):
    errors, observed, clip = run_model_sequence('IPSBiasedMF', kind, rank, clip='median', seed=1)
    _report(observed, 'clip %g %s rank %d' % (clip, kind, rank))
    assert not errors, errors[:6]
