"""Without a GPU: what the float64 comparison of the MF kernels (test_gpu_mf_reference.py) rests on.

- The float64 trainer (mf_reference.step) with biases, propensity and an acting clip, pinned to a torch float64 autograd
  model of the same step: (<p_u, q_i> + b_u + b_i + g) / max(prop_i, M), BaseModel.forward's BPR / MSE loss plus
  l2 * sum p^2, clip_grad_value_, then torch.optim.Adam / SGD / Adagrad with weight_decay = l2.
- The Python mirror of k_mf_step's pair -> (CTA, half-warp) map, pinned to dccf_mf_step_ctas, and the geometry and edge
  values each GPU case claims.
- Negative controls of the comparators: a float32 evaluation of the reference passes, and each defect a kernel could have
  is rejected."""
import numpy as np
import pytest
import torch

from dccf_b200 import _lib, build
from mf_reference import init_state, step
from test_gpu_mf_reference import (BIAS_CASES, BPR_P, COUNTS, EDGE_ITEMS, MSE_P, PAD, PAIRS_PER_CTA, STEP_CASES, UNIT, C,
                                   C_MODEL, check_bias, check_step, g_part_of, make_bias_problem, make_step_problem,
                                   pair_slots, row_sums_f32, loss_of, step_ctas)


@pytest.fixture(scope='module')
def lib():
    build.build()
    return _lib.load()


# ------------------------------------------------------------------------------------------------------------------
# the float64 trainer against torch autograd
# ------------------------------------------------------------------------------------------------------------------
def _torch_run(cls, kind, rank, clip, steps=4):
    U, I, P, lr, l2, M = 13, 17, 24, 0.05, 1e-3, 0.1
    rs = np.random.RandomState({'adam': 1, 'gd': 2, 'adagrad': 3}[kind] + 10 * rank)
    params = {'E_user': rs.standard_normal((U, 64)) * 0.3, 'E_item': rs.standard_normal((I, 64)) * 0.3,
              'user_bias': rs.standard_normal(U) * 0.3, 'item_bias': rs.standard_normal(I) * 0.3,
              'global_bias': np.asarray(0.1)}
    prop = None
    if cls == 'IPSBiasedMF':
        prop = rs.random_sample(I)
        prop[:4] = [0.0, M / 2, M, 1.0]
    tp = {k: torch.nn.Parameter(torch.tensor(v, dtype=torch.float64)) for k, v in params.items()}
    opt = {'adam': torch.optim.Adam, 'gd': torch.optim.SGD, 'adagrad': torch.optim.Adagrad}[kind](
        list(tp.values()), lr=lr, weight_decay=l2)
    hp = {'lr': lr, 'l2': l2, 'weight_decay': l2, 'clip': clip}
    state = init_state(params, kind)
    clipped = 0
    for t in range(1, steps + 1):
        X = np.stack([rs.randint(0, U, P), rs.randint(0, I, P)], 1).astype(np.int64)
        if rank == 1:
            X[P // 2:, 0] = X[:P // 2, 0]
            Y = np.r_[np.ones(P // 2), np.zeros(P // 2)]
        else:
            Y = rs.randint(1, 6, P).astype(np.float64)
        u, i = torch.from_numpy(X[:, 0]), torch.from_numpy(X[:, 1])
        opt.zero_grad()
        pred = (tp['E_user'][u] * tp['E_item'][i]).sum(1) + tp['user_bias'][u] + tp['item_bias'][i] + tp['global_bias']
        if prop is not None:
            pred = pred / torch.clamp(torch.from_numpy(prop)[i], min=M)
        if rank == 1:
            loss = -(pred[:P // 2] - pred[P // 2:]).sigmoid().log().sum()
        else:
            loss = torch.nn.MSELoss()(pred, torch.from_numpy(Y))
        (loss + l2 * sum((p ** 2).sum() for p in tp.values())).backward()
        clipped += sum(int((p.grad.abs() > clip).sum()) for p in tp.values())
        torch.nn.utils.clip_grad_value_(list(tp.values()), clip)
        opt.step()
        params, state, loss_ref, pred_ref, _ = step(params, state, t, X, Y, rank, hp, kind, prop=prop, M=M)
        assert float(loss.detach()) == pytest.approx(loss_ref, rel=1e-12, abs=1e-300), t
        assert np.abs(pred.detach().numpy() - pred_ref).max() <= 1e-12 * np.abs(pred_ref).max(), t
        for k, v in tp.items():
            got = v.detach().numpy()
            # (a step moves an element by up to lr: BPR's global-bias gradient is l2 terms plus cancelled rounding)
            assert np.abs(got - params[k]).max() <= 1e-11 * max(np.abs(params[k]).max(), lr), (t, k)
    return clipped


@pytest.mark.parametrize('clip', [50.0, 0.02])
@pytest.mark.parametrize('rank', [1, 0])
@pytest.mark.parametrize('kind', ['adam', 'gd', 'adagrad'])
@pytest.mark.parametrize('cls', ['IPSBiasedMF', 'BiasedMF'])
def test_reference_trainer_equals_torch_autograd(cls, kind, rank, clip):
    clipped = _torch_run(cls, kind, rank, clip)
    if clip < 1:
        assert clipped > 0                                  # the small clip acts


# ------------------------------------------------------------------------------------------------------------------
# geometry
# ------------------------------------------------------------------------------------------------------------------
def test_geometry_mirror_equals_the_library(lib):
    sizes = list(range(0, 2100)) + [65535, 65536, 65537, 10 ** 6 + 3, 2 ** 31 - 1]
    for P in sizes:
        assert lib.dccf_mf_step_ctas(P) == step_ctas(P), P
    for P in range(1, 600):
        for rank in (0, 1):
            if rank == 1 and P % 2:
                continue
            cta, hw = pair_slots(P, rank)
            assert cta.min() >= 0 and cta.max() == step_ctas(P) - 1 and hw.min() >= 0 and hw.max() < PAIRS_PER_CTA
            assert len(set(zip(cta, hw))) == P, (P, rank)          # one half-warp per pair
            if rank == 1:                                           # a BPR pair and its negative share a warp
                b = P // 2
                assert (cta[:b] == cta[b:]).all() and (hw[b:] == hw[:b] + 1).all() and (hw[:b] % 2 == 0).all()


def _margins(pb):
    c, ref = pb['case'], pb['ref']
    b = c.P // 2
    return ref['pred'][:b] - ref['pred'][b:]


def test_every_step_case_reaches_what_it_claims():
    seen = set()
    assert sorted(c.P for c in STEP_CASES if c.rank == 1 and c.cls == 'ips') == sorted(BPR_P)
    assert sorted(c.P for c in STEP_CASES if c.rank == 0 and c.cls == 'ips') == sorted(MSE_P)
    for c in STEP_CASES:
        pb = make_step_problem(c, STEP_CASES.index(c))
        cta, hw = pair_slots(c.P, c.rank)
        n = step_ctas(c.P)
        live_last = int((cta == n - 1).sum())
        seen.add(('last CTA live half-warps', live_last))
        if c.P % PAIRS_PER_CTA:
            seen.add('partial last CTA')
        if n > 1:
            seen.add('several CTAs')
        if (cta != np.arange(c.P) // PAIRS_PER_CTA).any():
            seen.add('pairs handled by a CTA other than their index CTA')
        if c.rank == 0 and c.P % 2:
            seen.add('odd MSE batch')
        if c.rank == 1 and c.P // 2 < 8:
            seen.add('short BPR batch')
        X, prop, M = pb['X'], pb['prop'], pb['M']
        p = prop[X[:, 1]]
        if c.cls == 'biased':
            assert (prop == 1).all() and M == 1.0
            seen.add('biased ' + ('bpr' if c.rank else 'mse'))
        else:
            for name, hit in (('prop 0', p == 0), ('prop below M', (p > 0) & (p < M)), ('prop M', p == np.float32(M)),
                              ('prop just above M', p == np.nextafter(np.float32(M), np.float32(2))),
                              ('prop 1', p == 1)):
                if hit.any():
                    seen.add(name)
        if c.rank == 1:
            x = _margins(pb)
            for name, hit in (('x = 0', x == 0), ('x > 88.7', x > 88.8), ('x < -88.7', x < -88.8),
                              ('87.3 < x < 88.7', (x > 87.4) & (x < 88.6)), ('|x| of order 1', np.abs(x) < 2)):
                if hit.any():
                    seen.add(name)
        else:
            if (pb['ref']['pred'] - pb['Y'] == 0).any():
                seen.add('e = 0')
        assert np.median(np.abs(pb['ref']['pred'])) > 0.1, c.name              # predictions of order 1
    for want in ('partial last CTA', 'several CTAs', 'pairs handled by a CTA other than their index CTA', 'odd MSE batch',
                 'short BPR batch', 'biased bpr', 'biased mse', 'prop 0', 'prop below M', 'prop M', 'prop just above M',
                 'prop 1', 'x = 0', 'x > 88.7', 'x < -88.7', '87.3 < x < 88.7', '|x| of order 1', 'e = 0'):
        assert want in seen, want
    # the last CTA with 1 and with 15 live half-warps, and full
    for k in (1, 2, 15, 16):
        assert ('last CTA live half-warps', k) in seen, k


def test_every_bias_case_reaches_what_it_claims():
    totals = set()
    for c in BIAS_CASES:
        pb = make_bias_problem(c)
        X = pb['X']
        for col, n_rows, hot in ((0, c.U, 'user'), (1, c.I, 'item')):
            counts = np.bincount(X[:, col], minlength=n_rows)
            if c.hot == hot:
                assert counts.max() == c.P and c.P <= 1024
            else:
                assert set(COUNTS) | {0} <= set(counts), (c.name, col)
        totals.add(c.U + c.I)
    assert {255, 256, 257} <= totals and min(totals) < 255 and max(totals) > 2 * 256


def test_every_hyper_parameter_term_is_visible():
    """At lr 0.05, l2 = wd = 1e-3 on parameters of order 0.1, the l2 and weight-decay terms move a parameter by many
    ulps; the bounds stay at or below 2^-16 relative."""
    p = np.float32(0.1)
    assert 0.05 * 1e-3 * p / np.spacing(p) > 100
    assert all(0 < c * UNIT <= 2.0 ** -16 for c in list(C.values()) + list(C_MODEL.values()))


# ------------------------------------------------------------------------------------------------------------------
# negative controls
# ------------------------------------------------------------------------------------------------------------------
def emulate_step(pb, defect=None):
    """A float32 evaluation of k_mf_step's outputs (numpy's own summation order), with one defect."""
    c, prm, X, Y = pb['case'], pb['prm'], pb['X'], pb['Y']
    P, f = c.P, np.float32
    u, i = X[:, 0], X[:, 1]
    pu, qi = prm['E_user'][u], prm['E_item'][i]
    with np.errstate(over='ignore', divide='ignore', invalid='ignore'):
        dot = (pu * qi).sum(1, dtype=np.float32)
        clamp = np.minimum if defect == 'fminf in the clamp' else np.maximum
        scale = clamp(pb['prop'][i], f(pb['M']))
        bias = prm['user_bias'][u] + prm['item_bias'][i] + prm['global_bias']
        if defect == 'bias added after the division':
            pred = (dot / scale + bias).astype(f)
        else:
            pred = ((dot + prm['user_bias'][u] + prm['item_bias'][i] + prm['global_bias']) / scale).astype(f)
        if c.rank == 1:
            b = P // 2
            neg = (np.arange(b) + b + (1 if defect == 'BPR negative from pair w + P/2 + 1' else 0)) % P
            x = pred[:b] - pred[neg]
            sig = (f(1) / (f(1) + np.exp(x))).astype(f)
            dl = np.concatenate([-sig, sig])
            t = np.where(x > 0, np.log1p(np.exp(-x)), np.log1p(np.exp(x)) - x).astype(f)
            term = np.concatenate([t, np.zeros(P - b, f)])
        else:
            e = pred - Y
            dl = (f(2) * e / f(P / 2 if defect == 'MSE divisor P/2' else P)).astype(f)
            term = (e * e).astype(f)
        r = dl if defect == 'r not divided by max(prop, M)' else (dl / scale).astype(f)
        gu, gi = r[:, None] * qi, r[:, None] * pu
    nan = lambda *s: np.full(s, np.nan, f)        # noqa: E731
    out = {'pred': nan(P + PAD), 'gb_rec': nan(P + PAD), 'gu_rec': nan(P + PAD, 64), 'gi_rec': nan(P + PAD, 64),
           'keys_u': np.full(P + PAD, -7, np.int32), 'keys_i': np.full(P + PAD, -7, np.int32)}
    out['pred'][:P], out['gb_rec'][:P], out['gu_rec'][:P], out['gi_rec'][:P] = pred, r, gu, gi
    out['keys_u'][:P], out['keys_i'][:P] = u, i
    n = step_ctas(P)
    out['g_part'], out['loss_part'] = nan(n + 4), nan(n + 4)
    out['g_part'][:n] = g_part_of(r, P, c.rank, drop_last=defect == 'g_part missing the last half-warp')
    cta, hw = pair_slots(P, c.rank)
    s = np.zeros((n, PAIRS_PER_CTA), f)
    s[cta, hw] = term
    acc = np.zeros(n, f)
    for k in range(PAIRS_PER_CTA):
        acc = (acc + s[:, k]).astype(f)
    out['loss_part'][:n] = acc
    return out


def emulate_bias(pb, defect=None):
    X, gb, U, I = pb['X'], pb['gb_rec'], pb['U'], pb['I']
    order = 'descending' if defect == 'bias records summed in descending order' else 'ascending'
    drop = defect == 'the first record of a row dropped'
    ku = X[:, 1] if defect == 'the user-bias record keyed to the item row' else X[:, 0]
    g_user = row_sums_f32(ku.astype(np.int32), gb, max(U, I), order, drop)[:U]
    g_item = row_sums_f32(X[:, 1].astype(np.int32), gb, I, order, drop)
    scale = 1.0 if defect == 'loss_scale not applied' else pb['loss_scale']
    return {'g_user': np.r_[g_user, np.full(5, np.nan, np.float32)], 'g_item': np.r_[g_item, np.full(5, np.nan, np.float32)],
            'loss': np.r_[loss_of(pb['loss_part'], scale), np.float32(np.nan)].astype(np.float32)}


def _step_fails(defect):
    total = 0
    for c in STEP_CASES:
        pb = make_step_problem(c, STEP_CASES.index(c))
        total += sum(check_step(pb, emulate_step(pb, defect), {}).values())
    return total


def _bias_fails(defect):
    total = 0
    for c in BIAS_CASES:
        pb = make_bias_problem(c, seed=1)
        total += sum(check_bias(pb, emulate_bias(pb, defect)).values())
    return total


def test_comparators_accept_a_float32_evaluation_of_the_reference():
    for c in STEP_CASES:
        pb = make_step_problem(c, STEP_CASES.index(c))
        observed = {}
        fails = check_step(pb, emulate_step(pb), observed)
        assert not any(fails.values()), (c.name, fails, observed)
    assert _bias_fails(None) == 0


STEP_DEFECTS = ['BPR negative from pair w + P/2 + 1', 'r not divided by max(prop, M)', 'fminf in the clamp',
                'bias added after the division', 'MSE divisor P/2', 'g_part missing the last half-warp']
BIAS_DEFECTS = ['bias records summed in descending order', 'the first record of a row dropped',
                'the user-bias record keyed to the item row', 'loss_scale not applied']


@pytest.mark.parametrize('defect', STEP_DEFECTS)
def test_step_comparator_rejects_a_defect(defect):
    assert _step_fails(defect) > 0


@pytest.mark.parametrize('defect', BIAS_DEFECTS)
def test_bias_comparator_rejects_a_defect(defect):
    assert _bias_fails(defect) > 0
