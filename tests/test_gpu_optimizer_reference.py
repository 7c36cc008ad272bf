"""The optimizer step (l2 + clip + weight decay + Adam / GD / Adagrad) against a float64 reference, element by element,
over its whole launch geometry.

The reference is a float64 restatement of what the kernels compute, fed the exact float32 values they read (parameters,
state, gradient records, dW / db partials):

    g = clip(sum of the row's records + 2 * l2 * p) + wd * p,  then the rule:
    Adam     torch's non-capturable _multi_tensor_adam with bias correction at step t
    GD       SGD, momentum 0
    Adagrad  lr_decay 0

What is compared is the UPDATE p_new - p_old and every state tensor, never the parameter norm-wise: at the step sizes
of a training run the update is a tiny fraction of p, and a norm-wise test on p cannot see the l2 / weight-decay terms.
The bound is |y_kernel - y_ref| <= C * 2^-20 * |y|_bound + ulp(y_kernel) / 2, where |y|_bound carries the input bounds
through each stage to first order (`reference` below); elements whose gradient lies within its own bound of +-clip may
clip either way.  Hyper-parameters are chosen so that every term moves p by many ulps.

Paths, for each rule: the unsplit dccf_adam_step; the split step driven from ids as DCCF._fused_split_step drives it
(dccf_adam_link_ids -> dccf_adam_untouched -> dccf_adam_csr_build -> dccf_adam_touched), with CSR ranges and with
linked lists, at every side-sweep width and the wide sweep; Adam's per-tensor entry points.  The test itself fills the
gradient records and the dW / db partials.  The case list states the geometry each case reaches;
test_optimizer_reference_cpu.py checks those claims against the library without a GPU."""
from collections import namedtuple

import numpy as np
import pytest
import torch

D = 64
U32 = 2.0 ** -24                 # unit roundoff of float32
UNIT = 2.0 ** -20
ETA = 2.0 ** -126                # a rounding below the normal range errs by up to 2^-150 absolute: 2^-126 in units of U32
# about 4 times the smallest C each output needed over this module on an NVIDIA B200 at a 1000 W power limit (p 0.044,
# m 0.050, v 0.037, s 0.048; the tests print them: "observed C")
C = {'p': 0.18, 'm': 0.2, 'v': 0.15, 's': 0.2}
RULES = {'adam': 0, 'gd': 1, 'adagrad': 2}
STATE = {'adam': ('m', 'v'), 'gd': (), 'adagrad': ('s',)}
LIST_CAP = 96                    # ADAM_LIST_CAP (adam.cu): longer lists take the fallback walk
WIDTHS = (32, 128, 224, 256, -1)  # side-sweep widths (0 = the library's default, 224) and the wide sweep
ADAM_STEPS = (1, 2, 3, 1000, 10 ** 6)


# ------------------------------------------------------------------------------------------------------------------
# launch geometry: Python mirror of marshal_adam's CTA assignment (adam.cu), pinned in test_optimizer_reference_cpu.py
# ------------------------------------------------------------------------------------------------------------------
def table_blocks(mode, n_rows, total_rows, n_rec, n_rec_all):
    if mode == 2:
        want = (n_rec + 15) // 16
        share = -(-(148 * 3 - 150) * n_rec // n_rec_all) if n_rec_all > 0 else 0
        want = min(want, share)
        return 1 if (want < 1 and n_rec > 0) else want
    budget = 148 if mode == 1 else 148 * 8
    want = (n_rows + 31) // 32
    share = -(-budget * n_rows // total_rows) if total_rows > 0 else 0
    want = min(want, share)
    return 1 if (want < 1 and n_rows > 0) else want


def dense_blocks(n):
    return min((n + 255) // 256, 148)


def blocks(mode, rows, recs, dense_n):
    """(block_lo, block_n) per tensor, tables first; grid size."""
    out, lo = [], 0
    for r, n in zip(rows, recs):
        b = table_blocks(mode, r, sum(rows), n, sum(recs))
        out.append((lo, b))
        lo += b
    for n in dense_n:
        b = dense_blocks(n)
        out.append((lo, b))
        lo += b
    return out, lo


def sweep_warps(mode, block_n, threads):
    """Warps a table's range holds in a sweep launch (modes 0, 1, 3)."""
    return block_n * ((256 if mode != 1 else threads) // 32)


# ------------------------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------------------------
# U, I: rows of the user / item table; P pairs of S sampled items per segment (item records P * (S + 1) per segment);
# n_seg record segments (data-parallel layout), user_seg >= 0: only that segment carries user records; pad: extra
# elements between segments; u_distinct: distinct user rows; i_counts: item rows planted with exactly these record
# counts; dense: (n, n_parts, part_stride - n) per dense tensor, the first is W [64, 64 + F] when F > 0 (its operand image
# is checked); edges: p = 0, |g| << eps, subnormal p, g = +-clip, +-inf and NaN elements; big_eps: eps large enough to tell
# sqrt(v) + eps from sqrt(v + eps); empty: rows of a third table without records; rules: the rules it runs.
Case = namedtuple('Case', 'name U I P S n_seg user_seg pad u_distinct i_counts dense F edges big_eps empty rules')
ALL = ('adam', 'gd', 'adagrad')
CASES = [
    Case('counts', 37, 1203, 150, 9, 1, -1, 0, 37, (1, 2, 3, 4, 5, 95, 96, 97, 700),
         ((64 * 832, 20, 37), (64, 20, 0)), 768, True, False, 1, ALL),
    Case('big_eps', 3, 1202, 64, 5, 1, -1, 0, 3, (2, 5), ((257, 17, 3), (255, 16, 0)), 0, False, True, 0, ALL),
    Case('hw_1', 1568, 30000, 1024, 10, 1, -1, 0, 1, (700,), ((1, 1, 0), (255, 15, 1)), 0, False, False, 0, ALL),
    Case('hw_stride', 2240, 74000, 1024, 10, 1, -1, 0, 400, (), ((64 * 2112, 60, 5), (64, 60, 0)), 2048, False, False,
         0, ALL),
    Case('hw_stride_1', 1568, 30000, 1024, 10, 1, -1, 0, 401, (3,), ((257, 33, 0), (64, 33, 7)), 0, False, False, 0,
         ALL),
    Case('hw_2stride', 2241, 74000, 1024, 10, 1, -1, 0, 800, (), ((255, 16, 0),), 0, False, False, 0, ALL),
    Case('hw_2stride_1', 1569, 30000, 1024, 10, 1, -1, 0, 801, (97,), ((64 * 832, 17, 0), (64, 17, 0)), 768, True,
         False, 3, ALL),
    Case('seg2', 501, 2003, 100, 4, 2, -1, 13, None, (96, 97), ((64 * 832, 2, 64), (64, 2, 0)), 768, True, False, 0,
         ALL),
    Case('seg8_user3', 130, 999, 40, 3, 8, 3, 5, None, (5, 95), ((257, 8, 9), (64, 8, 0)), 0, False, False, 0, ALL),
    Case('adam_steps', 33, 500, 32, 3, 1, -1, 0, None, (4,), ((255, 15, 0), (64, 15, 0)), 0, True, False, 0, ('adam',)),
]


def hyper(rule, big_eps=False, t=3):
    eps = {'adam': 1e-2, 'gd': 1e-8, 'adagrad': 1e-1}[rule] if big_eps else {'adam': 1e-8, 'gd': 1e-8, 'adagrad': 1e-10}[rule]
    return dict(rule=rule, lr=0.1, l2=0.05, wd=0.02, clip=None, eps=eps, beta1=0.85, beta2=0.995, t=t)


def records_of(c):
    """Global record counts (user, item) of a case."""
    Z = c.S + 1
    n_u = c.P if c.user_seg >= 0 else c.n_seg * c.P
    return n_u, c.n_seg * c.P * Z


# ------------------------------------------------------------------------------------------------------------------
# problem
# ------------------------------------------------------------------------------------------------------------------
def _plant(rs, n_rows, n_rec, counts):
    """n_rec keys over n_rows rows with one row per planted count holding exactly that many records."""
    rows = rs.permutation(n_rows)
    planted, rest = rows[:len(counts)], rows[len(counts):]
    keys = np.concatenate([np.full(k, r) for r, k in zip(planted, counts)] +
                          [rs.choice(rest, size=n_rec - sum(counts))]) if n_rec > sum(counts) else \
        np.concatenate([np.full(k, r) for r, k in zip(planted, counts)])
    assert len(keys) == n_rec
    return keys[rs.permutation(n_rec)].astype(np.int32)


def _distinct(rs, n_rows, n_rec, k):
    rows = rs.permutation(n_rows)[:k]
    keys = np.concatenate([rows, rs.choice(rows, size=n_rec - k)])
    return keys[rs.permutation(n_rec)].astype(np.int32)


def make_problem(c, rule, seed=0, big_eps=None):
    rs = np.random.RandomState(seed)
    hp = hyper(rule, c.big_eps if big_eps is None else big_eps)
    Z = c.S + 1
    n_u, n_i = records_of(c)
    ku = _distinct(rs, c.U, n_u, c.u_distinct) if c.u_distinct else rs.randint(0, c.U, n_u).astype(np.int32)
    ki = _plant(rs, c.I, n_i, c.i_counts)
    gu = rs.standard_normal((n_u, D)).astype(np.float32)
    gi = rs.standard_normal((n_i, D)).astype(np.float32)
    # ids of each segment as dccf_adam_link_ids reads them: X [P, 2] then sample_item [P, S], seg_stride apart
    seg_stride = 2 * c.P + c.P * c.S + c.pad
    ids = rs.randint(0, min(c.U, c.I), (c.n_seg, seg_stride)).astype(np.int64)
    for s in range(c.n_seg):
        X = ids[s, :2 * c.P].reshape(c.P, 2)
        si = ids[s, 2 * c.P:2 * c.P + c.P * c.S].reshape(c.P, c.S)
        kseg = ki[s * c.P * Z:(s + 1) * c.P * Z].reshape(c.P, Z)
        X[:, 1] = kseg[:, 0]
        si[:] = kseg[:, 1:]
        if c.user_seg < 0:
            X[:, 0] = ku[s * c.P:(s + 1) * c.P]
        elif s == c.user_seg:
            X[:, 0] = ku
        else:
            X[:, 0] = rs.randint(0, c.U, c.P)

    def table(n_rows, keys, grads, n_seg, seg_len):
        p = (rs.standard_normal((n_rows, D)) * 2).astype(np.float32)
        st = {}
        if rule == 'adam':
            st['m'] = (rs.standard_normal((n_rows, D)) * 0.5).astype(np.float32)
            st['v'] = (np.abs(rs.standard_normal((n_rows, D))) * 0.5).astype(np.float32)
        elif rule == 'adagrad':
            st['s'] = (np.abs(rs.standard_normal((n_rows, D))) * 0.5).astype(np.float32)
        return dict(n_rows=n_rows, p=p, st=st, keys=keys, grads=grads, n_seg=n_seg, seg_len=seg_len)

    tables = [table(c.U, ku, gu, 1 if c.user_seg >= 0 else c.n_seg, c.P),
              table(c.I, ki, gi, c.n_seg, c.P * Z)]
    if c.empty:
        tables.append(table(c.empty, np.zeros(0, np.int32), np.zeros((0, D), np.float32), 0, 0))
    dense = []
    for n, n_parts, extra in c.dense:
        parts = (rs.standard_normal((n_parts, n)) / np.sqrt(n_parts)).astype(np.float32)
        d = dict(n=n, n_parts=n_parts, stride=n + extra, parts=parts, p=(rs.standard_normal(n) * 2).astype(np.float32))
        d['st'] = {k: (v.reshape(-1)[:n].copy() if v.size >= n else np.resize(v.reshape(-1), n))
                   for k, v in tables[0]['st'].items()}
        dense.append(d)
    # the clip near the 70th percentile of |g| (so that some elements clip only because of the l2 term)
    g1 = np.concatenate([(row_sums(t)[0] + 2 * np.float32(hp['l2']) * t['p'].astype(np.float64)).ravel() for t in tables[:2]])
    hp['clip'] = float(np.float32(np.percentile(np.abs(g1), 70)))
    if c.edges:
        _edges(rs, tables, dense, hp, rule)
    return dict(case=c, hp=hp, ids=ids, seg_stride=seg_stride, tables=tables, dense=dense)


def _edges(rs, tables, dense, hp, rule):
    """p = 0 with zero state (0 / eps), |g| << eps, subnormal p (and g), g exactly +-clip, +-inf and NaN elements."""
    clip = np.float32(hp['clip'])
    for t in tables[:2]:
        counts = np.bincount(t['keys'], minlength=t['n_rows'])
        untouched, single = np.flatnonzero(counts == 0), np.flatnonzero(counts == 1)
        multi = np.flatnonzero(counts >= 3)
        t['p'][untouched[:3]] = 0
        for v in t['st'].values():
            v[untouched[:3]] = 0
        t['p'][untouched[3:5]] = (rs.standard_normal((len(untouched[3:5]), D)) * 1e-12).astype(np.float32)
        for v in t['st'].values():
            v[untouched[3:5]] = 0
        t['p'][untouched[5:7]] = (rs.standard_normal((len(untouched[5:7]), D)) * 1e-39).astype(np.float32)
        if len(single) < 3:
            continue
        rec = lambda row: int(np.flatnonzero(t['keys'] == row)[0])       # noqa: E731
        a, b, n = single[0], single[1], single[2]
        t['p'][a] = 0                                                     # g = +-clip exactly
        t['grads'][rec(a), :8], t['grads'][rec(a), 8:16] = clip, -clip
        t['grads'][rec(b), 0], t['grads'][rec(b), 1] = np.inf, -np.inf   # +-inf
        t['grads'][rec(n), 5] = np.nan                                    # NaN from a single record
        if len(multi):
            t['grads'][np.flatnonzero(t['keys'] == multi[0])[-1], 9] = np.nan   # NaN in a longer list
    d = dense[0]
    d['parts'][d['n_parts'] - 1, d['n'] // 2] = np.nan
    if d['n'] > 1:
        d['parts'][0, 0] = np.inf


def row_sums(t):
    """float64 sum of each row's records, and the bound of the float32 ascending sum: (n - 1) * sum |rec|."""
    n_rows = t['n_rows']
    g = np.zeros((n_rows, D))
    a = np.zeros((n_rows, D))
    with np.errstate(invalid='ignore', over='ignore'):
        np.add.at(g, t['keys'], t['grads'].astype(np.float64))
        np.add.at(a, t['keys'], np.abs(t['grads'].astype(np.float64)))
        n = np.bincount(t['keys'], minlength=n_rows)[:, None]
        return g, np.where(n > 1, (n - 1) * a, 0.0), n


def dense_sums(d):
    parts = d['parts'].astype(np.float64)
    with np.errstate(invalid='ignore', over='ignore'):
        return parts.sum(0), np.where(d['n_parts'] > 1, (d['n_parts'] - 1) * np.abs(parts).sum(0), 0.0)


# ------------------------------------------------------------------------------------------------------------------
# float64 reference with first-order bounds: every A_x below satisfies |x_float32_path - x| <~ U32 * A_x.  Each rounding
# adds U32 * |result| relative and, for results in the subnormal range, ETA absolute (a parameter that decays towards zero
# under the regulariser alone gets there within a few Adagrad steps)
# ------------------------------------------------------------------------------------------------------------------
def _sqrt_bound(A, x):
    with np.errstate(divide='ignore', invalid='ignore'):
        return np.minimum(np.where(x > 0, A / (2 * np.sqrt(np.maximum(x, 0))), np.inf), np.sqrt(A / U32))


def reference(hp, p, st, gs, A_gs, flip=None, defect=None):
    """Update and new state of one tensor.  p, st: float32 inputs; gs, A_gs: float64 gradient sum and its bound.
    flip: elements that take the other side of the clip.  defect: a deliberate error (negative controls)."""
    f32 = lambda x: float(np.float32(x))        # noqa: E731   the scalars the kernel reads as float
    l2, wd, clip, eps = f32(hp['l2']), f32(hp['wd']), f32(hp['clip']), f32(hp['eps'])
    lr, rule = hp['lr'], hp['rule']
    if defect == 'l2 and wd swapped':
        l2, wd = wd, l2
    if defect == 'no weight decay':
        wd = 0.0
    p = p.astype(np.float64)
    with np.errstate(invalid='ignore', over='ignore', divide='ignore'):
        g1 = gs + 2 * l2 * p
        A1 = A_gs + np.abs(2 * l2 * p) + np.abs(g1) + 2 * ETA
        if defect == 'clip before + 2*l2*p':
            g1 = np.clip(gs, -clip, clip) + 2 * l2 * p
        over = np.abs(g1) > clip
        if flip is not None:
            over = over ^ flip
        g2 = np.where(over, np.sign(g1) * clip, g1)
        A2 = np.where(over, 0.0, A1)
        if defect == 'clip before + 2*l2*p':
            g2, A2 = g1, A1
        if defect == 'NaN clipped to -clip':
            g2 = np.where(np.isnan(g2), -clip, g2)
        g3 = g2 + wd * p
        if defect == 'clip after + wd*p':
            g3 = np.clip(g1 + wd * p, -clip, clip)
        A3 = A2 + np.abs(g3) + ETA
        out = {'g1': g1, 'A_g1': A1}
        if rule == 'gd':
            dp = -lr * g3
            out.update(p=dp, A_p=lr * A3 + np.abs(dp))
        elif rule == 'adagrad':
            s = st['s'].astype(np.float64) + g3 * g3
            A_s = 2 * np.abs(g3) * A3 + np.abs(s) + ETA
            sq = np.sqrt(s)
            A_sq = _sqrt_bound(A_s, s) + 2 * sq
            std = sq + eps
            q = g3 / std
            A_q = A3 / std + np.abs(g3) * (A_sq + std) / std ** 2 + 2 * np.abs(q) + ETA
            dp = -lr * q
            out.update(p=dp, A_p=lr * A_q + np.abs(dp), s=s, A_s=A_s)
        else:
            b1, b2, t = hp['beta1'], hp['beta2'], hp['t']
            if defect == 'bias correction at t - 1':
                t = t - 1
            bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
            m0, v0 = st['m'].astype(np.float64), st['v'].astype(np.float64)
            m = b1 * m0 + (1 - b1) * g3
            A_m = (1 - b1) * (A3 + 2 * np.abs(g3 - m0)) + np.abs(m) + 2 * ETA
            v = b2 * v0 + (1 - b2) * g3 * g3
            A_v = 2 * b2 * np.abs(v0) + (1 - b2) * (3 * g3 * g3 + 2 * np.abs(g3) * A3) + np.abs(v) + 2 * ETA
            ib = 1 / np.sqrt(bc2) if bc2 > 0 else np.inf
            sq = np.sqrt(v)
            A_sq = _sqrt_bound(A_v, v) + 2 * sq
            den = np.sqrt(v / bc2 + eps) if defect == 'eps inside the square root' else sq * ib + eps
            A_den = ib * (A_sq + sq) + den
            q = m / den
            A_q = A_m / den + np.abs(m) * A_den / den ** 2 + 2 * np.abs(q) + ETA
            step = lr / bc1
            dp = -step * q
            out.update(p=dp, A_p=step * A_q + np.abs(dp), m=m, A_m=A_m, v=v, A_v=A_v)
    return out


def _check(got, ref, A, ulp_of, c):
    """(failing elements, smallest C each element needs)."""
    half = 0.5 * np.spacing(np.abs(ulp_of.astype(np.float32))).astype(np.float64)
    nan_ref = np.isnan(ref)
    with np.errstate(invalid='ignore', over='ignore', divide='ignore'):
        d = np.abs(got - ref)
        bad = (nan_ref != np.isnan(got)) | (~nan_ref & ~(d <= c * UNIT * A + half))
        need = np.where(nan_ref, 0.0, np.where(d <= half, 0.0, (d - half) / (UNIT * A)))
    return bad, np.nan_to_num(need, nan=np.inf)


def compare(rule, hp, p_old, st_old, gs, A_gs, got, cs=None, defect=None):
    """got: {'p': p_new, state...} float32 from a kernel.  Returns ({output: number of failing elements}, {output:
    largest C needed}) over the tensor; the update is compared as p_new - p_old."""
    cs = C if cs is None else cs
    outs = ('p',) + STATE[rule]

    def judge(ref):
        res = {}
        for k in outs:
            if k == 'p':
                y, y_ref, ulp_of = got['p'].astype(np.float64) - p_old.astype(np.float64), ref['p'], got['p']
            else:
                y, y_ref, ulp_of = got[k].astype(np.float64), ref[k], got[k]
            res[k] = _check(y, y_ref, ref['A_' + k], ulp_of, cs[k])
        return res

    ref = reference(hp, p_old, st_old, gs, A_gs, defect=defect)
    a = judge(ref)
    # the clip's kink: within its own bound of +-clip the gradient may clip either way
    with np.errstate(invalid='ignore'):
        amb = np.isfinite(ref['g1']) & (np.abs(np.abs(ref['g1']) - np.float32(hp['clip'])) <= cs['p'] * UNIT * ref['A_g1'])
    bad_a = np.any([a[k][0] for k in outs], axis=0)
    if amb.any():
        b = judge(reference(hp, p_old, st_old, gs, A_gs, flip=amb, defect=defect))
        bad_b = np.any([b[k][0] for k in outs], axis=0)
        take_b = amb & bad_a & ~bad_b
        bad = bad_a & ~take_b
        need = {k: np.where(take_b, b[k][1], a[k][1]) for k in outs}
    else:
        bad, need = bad_a, {k: a[k][1] for k in outs}
    fails = {k: int((bad & a[k][0]).sum()) if amb.any() else int(a[k][0].sum()) for k in outs}
    fails['any'] = int(bad.sum())
    return fails, {k: float(need[k].max()) if need[k].size else 0.0 for k in outs}


def check_problem(pb, got, observed, where, defect=None):
    """Every table and dense tensor of a problem against the reference; records the C each output needed."""
    hp, rule = pb['hp'], pb['hp']['rule']
    errors = []
    items = [(t, row_sums(t)[:2]) for t in pb['tables']] + [(d, dense_sums(d)) for d in pb['dense']]
    for i, (x, (gs, A)) in enumerate(items):
        g = {k: v.reshape(x['p'].shape) for k, v in got[i].items()}
        fails, need = compare(rule, hp, x['p'], x['st'], gs, A, g, defect=defect)
        for k, v in need.items():
            observed[k] = max(observed.get(k, 0.0), v)
        if fails['any']:
            errors.append((where, i, fails, need))
    return errors


# ------------------------------------------------------------------------------------------------------------------
# device runs
# ------------------------------------------------------------------------------------------------------------------
def _dev(pb):
    """Fresh device copies of a problem's tensors and record buffers in their segmented layout."""
    c = pb['case']
    out = {'tables': [], 'dense': []}
    for t in pb['tables']:
        n_rec = len(t['keys'])
        seg_len = max(t['seg_len'], 1)
        kstride = seg_len + (c.pad if t['n_seg'] > 1 else 0)
        keys = np.zeros((max(t['n_seg'], 1), kstride), np.int32)
        grads = np.full((max(t['n_seg'], 1), kstride, D), 1e3, np.float32)       # the padding must never be read
        for s in range(t['n_seg']):
            keys[s, :seg_len] = t['keys'][s * seg_len:(s + 1) * seg_len]
            grads[s, :seg_len] = t['grads'][s * seg_len:(s + 1) * seg_len]
        dt = dict(p=torch.from_numpy(t['p']).cuda(), st={k: torch.from_numpy(v).cuda() for k, v in t['st'].items()},
                  keys=torch.from_numpy(keys).cuda(), grads=torch.from_numpy(grads).cuda(), n_rec=n_rec,
                  n_seg=t['n_seg'], seg_len=t['seg_len'], kstride=kstride,
                  head=torch.full((t['n_rows'],), -1, dtype=torch.int32, device='cuda'),
                  next=torch.full((max(n_rec, 1),), 7, dtype=torch.int32, device='cuda'))
        out['tables'].append(dt)
    for d in pb['dense']:
        parts = np.full((d['n_parts'], d['stride']), 1e3, np.float32)
        parts[:, :d['n']] = d['parts']
        out['dense'].append(dict(p=torch.from_numpy(d['p']).cuda(), st={k: torch.from_numpy(v).cuda() for k, v in d['st'].items()},
                                 parts=torch.from_numpy(parts).cuda(), n_parts=d['n_parts'], stride=d['stride']))
    return out


def _mv(x):
    return (x['st'].get('m', x['st'].get('s')), x['st'].get('v'))


def _descr(dv, csr):
    from dccf_b200 import kernels
    tables = []
    for i, t in enumerate(dv['tables']):
        bufs = None
        if csr and t['n_rec'] > 0:
            t['csr'] = bufs = (torch.full((t['n_rec'],), -5, dtype=torch.int32, device='cuda'),
                               torch.full((t['p'].shape[0],), -5, dtype=torch.int32, device='cuda'),
                               torch.full((2 * t['n_rec'],), -5, dtype=torch.int32, device='cuda'),
                               torch.zeros(2, dtype=torch.int32, device='cuda'))
        tables.append(kernels.adam_table(t['p'], *_mv(t), t['keys'], t['grads'], t['n_seg'], t['seg_len'],
                                         t['kstride'], t['kstride'] * D, t['head'], t['next'], csr=bufs))
    dense = [kernels.adam_tensor(d['p'], *_mv(d), d['parts'], d['n_parts'], d['stride']) for d in dv['dense']]
    return tables, dense


def _hp(pb, t=None, step_dev=None):
    from dccf_b200 import kernels
    h = pb['hp']
    return kernels.make_adam(h['lr'], h['l2'], h['wd'], step=h['t'] if t is None else t, step_dev=step_dev,
                             beta1=h['beta1'], beta2=h['beta2'], eps=h['eps'], clip=h['clip'], rule=RULES[h['rule']])


def _read(dv):
    torch.cuda.synchronize()
    return [dict({'p': x['p'].cpu().numpy()}, **{k: v.cpu().numpy() for k, v in x['st'].items()})
            for x in dv['tables'] + dv['dense']]


def _heads_released(dv):
    return all(int((t['head'] != -1).sum()) == 0 for t in dv['tables'])


def run_all(pb, step_dev_t=None):
    """dccf_adam_step: k_link_all + k_*_all."""
    from dccf_b200 import kernels
    dv = _dev(pb)
    tables, dense = _descr(dv, False)
    sd = torch.tensor([step_dev_t], dtype=torch.int32, device='cuda') if step_dev_t is not None else None
    kernels.adam_step(tables, dense, _hp(pb, step_dev=sd))
    out = _read(dv)
    assert _heads_released(dv)
    return out


def run_split(pb, csr=True, threads=0, step_dev_t=None):
    """The split step as DCCF._fused_split_step drives it: link from the ids (counting mode with CSR), the
    untouched-row sweep, the CSR build, the touched-row sweep with W's image and the device counters."""
    from dccf_b200 import kernels
    c, rule = pb['case'], pb['hp']['rule']
    dv = _dev(pb)
    tables, dense = _descr(dv, csr)
    tu, ti = dv['tables'][0], dv['tables'][1]
    ids = torch.from_numpy(pb['ids']).cuda().view(-1)
    dims = kernels.make_dims(c.U, c.I, 64, c.S, 1)
    extra = kernels.make_link_extra(rec_rows=(tu['csr'][0], ti['csr'][0])) if csr else None
    kernels.adam_link_ids(dims, ids, ids[2 * c.P:], tu['head'], tu['next'], ti['head'], ti['next'], n_pairs=c.P,
                          n_seg=c.n_seg, seg_stride=pb['seg_stride'] if c.n_seg > 1 else 0, user_seg=c.user_seg,
                          extra=extra)
    sd = torch.tensor([step_dev_t], dtype=torch.int32, device='cuda') if step_dev_t is not None else None
    hp = _hp(pb, step_dev=sd)
    kernels.adam_untouched(tables, hp, threads)
    if csr:
        kernels.adam_csr_build(tables)
    counter = torch.zeros(1, dtype=torch.int32, device='cuda')
    offset = torch.full((1,), 11, dtype=torch.int64, device='cuda')
    cursor = torch.full((1,), 5, dtype=torch.int64, device='cuda')
    wimg, K = None, 0
    if c.F:
        K = 64 + c.F
        wimg = torch.zeros(kernels.train_w_image_floats(c.F), dtype=torch.float32, device='cuda')
    kernels.adam_touched(tables, dense, hp, True, wimg, 0, K, counter, sd, offset, advance_cursor_dev=cursor)
    out = _read(dv)
    # post-conditions: lists released, counters advanced by exactly one, the CTA counter back at zero
    assert _heads_released(dv)
    if csr:
        assert all(int(t['csr'][3].abs().sum()) == 0 for t in dv['tables'] if 'csr' in t)
    assert int(counter) == 0 and int(offset) == 12 and int(cursor) == 6
    if sd is not None:
        assert int(sd) == step_dev_t + 1
    if wimg is not None:
        want = torch.empty_like(wimg)
        kernels.train_prep_w_image(dv['dense'][0]['p'], c.F, want)
        torch.cuda.synchronize()
        assert torch.equal(wimg.view(torch.int32), want.view(torch.int32)), 'W image != dccf_train_prep_w_image(W_new)'
    return out


def run_per_tensor(pb):
    """Adam's per-tensor entry points: dccf_adam_sweep_seg (dccf_adam_sweep for one segment) and dccf_adam_dense."""
    from dccf_b200 import kernels
    dv = _dev(pb)
    hp = _hp(pb)
    for t in dv['tables']:
        m, v = t['st']['m'], t['st']['v']
        if t['n_seg'] == 1:
            kernels.adam_sweep(t['p'], m, v, t['keys'], t['grads'], t['n_rec'], t['head'], t['next'], hp)
        else:
            kernels.adam_sweep_seg(t['p'], m, v, t['keys'], t['grads'], t['n_seg'], t['seg_len'], t['kstride'],
                                   t['kstride'] * D, t['head'], t['next'], hp)
    for d in dv['dense']:
        kernels.adam_dense(d['p'], d['st']['m'], d['st']['v'], d['parts'], d['n_parts'], d['stride'], hp)
    out = _read(dv)
    assert _heads_released(dv)
    return out


def _same(a, b):
    return all(np.array_equal(x[k].view(np.int32), y[k].view(np.int32)) for x, y in zip(a, b) for k in x)


def _report(observed, name):
    print('observed C %s: %s' % (name, ', '.join('%s %.3g' % kv for kv in sorted(observed.items()))))


pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('case', CASES, ids=[c.name for c in CASES])
def test_optimizer_step_against_float64_reference(case):
    """Every rule of the case on dccf_adam_step and on the split step (CSR and lists, every sweep width), against the
    reference, plus the bitwise invariants between the paths."""
    errors, observed = [], {}
    for rule in case.rules:
        pb = make_problem(case, rule, seed=CASES.index(case))
        ref_all = run_all(pb)
        errors += check_problem(pb, ref_all, observed, (rule, 'all'))
        csr = run_split(pb, csr=True, threads=0)
        errors += check_problem(pb, csr, observed, (rule, 'csr'))
        assert _same(ref_all, csr), (rule, 'k_*_all != split step')
        assert _same(csr, run_split(pb, csr=True, threads=0)), (rule, 'two runs differ')
        assert _same(csr, run_split(pb, csr=False, threads=0)), (rule, 'CSR != linked lists')
        for w in WIDTHS:
            assert _same(csr, run_split(pb, csr=True, threads=w)), (rule, 'sweep width %d' % w)
        if rule == 'adam':
            per = run_per_tensor(pb)
            errors += check_problem(pb, per, observed, (rule, 'per-tensor'))
    _report(observed, case.name)
    assert not errors, errors[:6]


@pytest.mark.parametrize('t', ADAM_STEPS)
def test_adam_step_number_host_and_device(t):
    """Adam's bias correction at t in {1, 2, 3, 1000, 10^6}: host step and step_dev give the same bits, on the unsplit and
    the split step, and both match the reference at t."""
    case = [c for c in CASES if c.name == 'adam_steps'][0]
    pb = make_problem(case, 'adam', seed=t % 97)
    pb['hp']['t'] = t
    observed, errors = {}, []
    host = run_all(pb)
    errors += check_problem(pb, host, observed, ('all', t))
    assert _same(host, run_all(pb, step_dev_t=t))
    split = run_split(pb, step_dev_t=t)
    assert _same(host, split)
    errors += check_problem(pb, split, observed, ('split', t))
    _report(observed, 't=%d' % t)
    assert not errors, errors[:6]


def test_nan_gradient_stays_nan():
    """A NaN gradient element gives NaN in p and in every state tensor of its element (clip_grad_value_ keeps NaN),
    on every rule and path; its neighbours stay finite."""
    case = [c for c in CASES if c.name == 'counts'][0]
    for rule in ALL:
        pb = make_problem(case, rule)
        t = pb['tables'][1]
        row = int(t['keys'][np.flatnonzero(np.isnan(t['grads'][:, 5]))[0]])
        for where, out in (('all', run_all(pb)), ('split', run_split(pb))):
            got = out[1]
            for k in got:
                assert np.isnan(got[k][row, 5]), (rule, where, k)
                assert np.isfinite(got[k][row, 4]) and np.isfinite(got[k][row, 6]), (rule, where, k)


# ------------------------------------------------------------------------------------------------------------------
# the step's own wiring: the whole model, its descriptors, its step numbers
# ------------------------------------------------------------------------------------------------------------------
def _snapshot(model):
    opt = model.optimizer
    params = {k: p.data.detach().cpu().numpy().copy() for k, p in opt.params.items()}
    st = {k: dict(zip(STATE[opt.kind], [x.cpu().numpy().copy() for x in opt.state_of(k) if x is not None]))
          for k in opt.params}
    return params, st


def _model_update_errors(model, before, t, users, observed):
    """The update of the step just taken, recomputed in float64 from the gradient records and dW / db partials it left in
    the model's workspace.  before: _snapshot() taken before the step; t: its step number; users: the user ids of its
    batch (the user records must be those of this batch)."""
    from dccf_b200 import kernels
    opt, ws = model.optimizer, model._ws
    P, S, A = len(users), model.sample_num, model.attribute_num
    Z, F = S + 1, model.feature_embedding.shape[1]
    recs = {'E_user': (ws['keys_u'][:P].cpu().numpy(), ws['gu_rec'][:P * D].view(P, D).cpu().numpy()),
            'E_item': (ws['keys_i'][:P * Z].cpu().numpy(), ws['gi_rec'][:P * Z * D].view(P * Z, D).cpu().numpy())}
    assert (recs['E_user'][0] == users).all(), t
    hp = dict(rule=opt.kind, lr=opt.lr, l2=opt.l2, wd=opt.weight_decay, clip=opt.clip, eps=opt.eps, beta1=opt.beta1,
              beta2=opt.beta2, t=t)
    (p0, s0), (p1, s1) = before, _snapshot(model)
    errors = []
    for k in opt.params:
        if k in recs:
            gs, A_gs, _ = row_sums(dict(n_rows=p0[k].shape[0], keys=recs[k][0], grads=recs[k][1]))
        else:
            n_parts, n = kernels.train_bwd_splits(P * Z * A, F), p0[k].size
            parts = (ws['gW_part'] if k == 'W' else ws['gb_part'])[:n_parts * n].cpu().numpy().reshape(n_parts, n)
            gs, A_gs = (x.reshape(p0[k].shape) for x in dense_sums(dict(parts=parts, n_parts=n_parts)))
        fails, need = compare(opt.kind, hp, p0[k], s0[k], gs, A_gs, dict({'p': p1[k]}, **s1[k]))
        for o, v in need.items():
            observed[o] = max(observed.get(o, 0.0), v)
        if fails['any']:
            errors.append((t, k, fails, need))
    return errors


@pytest.mark.parametrize('kind', ALL)
@pytest.mark.parametrize('rank', [1, 0])
def test_model_steps_against_float64_reference(kind, rank):
    """DCCF.train_step with a visible lr / l2: two eager steps, three graph replays, then a device-resident epoch of four
    batches (the first eager, then one launch of the staged graph per batch).  Before each step the parameters and the
    state are snapshot; after it the step's gradient records and dW / db partials are read from the model's workspace and
    the update is recomputed in float64.  Checks the descriptors _step_tables builds (counts, strides, partial counts),
    that every step, replays and epoch launches included, uses its own step number, and that the staged graph reads
    batch b (ids, and labels at rank 0) and leaves the batch cursor at b + 1."""
    from test_gpu_parity import make_model, random_problem
    U, I, F, P, S, A = 60, 90, 768, 64, 5, 2
    params, X, si, _, _ = random_problem(5, U, I, F, P, S, A, 0.0, 0.0)
    model = make_model(params, S, A, 0.1)
    model.optimizer = model.make_fused_optimizer(lr=0.1, l2=0.01, kind=kind)
    opt = model.optimizer
    rs = np.random.RandomState(2)
    n_batches = 9

    def batch(b):
        Xb = np.roll(X, 7 * b, axis=0).copy()
        Xb[P // 2:, 0] = Xb[:P // 2, 0]           # users with two records
        return Xb, np.roll(si, b, axis=0).copy(), rs.random_sample(P).astype(np.float32)
    batches = [batch(b) for b in range(n_batches)]
    observed, errors = {}, []
    t = 0
    for b in range(5):
        model.use_cuda_graph = b >= 2
        Xb, sib, Yb = batches[b]
        before = _snapshot(model)
        model.train_step({'X': torch.from_numpy(Xb).cuda(), 'rank': rank, 'train': True, 'dropout': 0.2,
                          'Y': torch.from_numpy(Yb).cuda(), 'sample_item': torch.from_numpy(sib)})
        torch.cuda.synchronize()
        t += 1
        assert opt.step_count == t
        errors += _model_update_errors(model, before, t, Xb[:, 0], observed)
    # the device-resident epoch: the remaining batches
    epoch = batches[5:]
    X_ep = torch.from_numpy(np.stack([e[0] for e in epoch])).cuda()
    si_ep = torch.from_numpy(np.stack([e[1] for e in epoch])).cuda()
    Y_ep = torch.from_numpy(np.stack([e[2] for e in epoch])).cuda() if rank == 0 else None
    before = _snapshot(model)
    step = model.begin_resident_epoch(X_ep, si_ep, 0.2, Y_epoch=Y_ep)
    assert step is not None and step.remaining() == len(epoch) - 1
    torch.cuda.synchronize()
    t += 1
    errors += _model_update_errors(model, before, t, epoch[0][0][:, 0], observed)
    g = [v for k, v in model._graphs.items() if k[4]][0]          # the staged graph
    for b in range(1, len(epoch)):
        before = _snapshot(model)
        step()
        torch.cuda.synchronize()
        t += 1
        assert opt.step_count == t and int(g['step_dev']) == t + 1 and int(g['cursor']) == b + 1, (b, t)
        assert torch.equal(g['X'], X_ep[b]) and torch.equal(g['si'], si_ep[b]), b
        if rank == 0:
            assert torch.equal(g['Y'], Y_ep[b]), b
        errors += _model_update_errors(model, before, t, epoch[b][0][:, 0], observed)
    with pytest.raises(StopIteration):
        step()
    _report(observed, 'model %s rank %d' % (kind, rank))
    assert not errors, errors[:6]
