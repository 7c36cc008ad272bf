"""Float64 NumPy reference of one BiasedMF / IPSBiasedMF training step (the semantics of BaseModel.forward +
BaseRunner.fit's step, src/runners/BaseRunner.py:175-188):

    pred = (<p_u, q_i> + b_u + b_i + g) / max(prop_i, M)         (biases=False: <p_u, q_i> only, RecModel)
    loss = sum_j -log sigmoid(pred_j - pred_{j+P/2})  (rank 1)   or   mean_p (pred_p - Y_p)^2  (rank 0)
    grad = clamp(d loss / d p + 2 l2 p, -clip, clip) + wd p, then Adam / GD / Adagrad on every element

Besides the result it returns the first-order magnitudes the GPU comparison needs: for every gradient element the sum of
the absolute values of the terms it is made of (`abs` dict), so that an fp32 evaluation differs from the result by at
most C * 2^-20 times that magnitude."""
import numpy as np

PARAMS = ('E_user', 'E_item', 'user_bias', 'item_bias', 'global_bias')


def init_state(params, kind):
    if kind == 'adam':
        return {k: {'m': np.zeros_like(v), 'v': np.zeros_like(v)} for k, v in params.items()}
    if kind == 'adagrad':
        return {k: {'s': np.zeros_like(v)} for k, v in params.items()}
    return {k: {} for k in params}


def forward(params, X, prop=None, M=1.0, biases=True):
    """(pred [P], scale [P], |terms| of pred [P]) in float64."""
    u, i = X[:, 0], X[:, 1]
    pu, qi = params['E_user'][u], params['E_item'][i]
    pred = (pu * qi).sum(1)
    mag = np.abs(pu * qi).sum(1)
    if biases:
        bu, bi, g = params['user_bias'][u], params['item_bias'][i], params['global_bias']
        pred = pred + bu + bi + g
        mag = mag + np.abs(bu) + np.abs(bi) + np.abs(g)
    s = np.ones(len(X)) if prop is None else np.maximum(np.asarray(prop, np.float64)[i], M)
    return pred / s, s, mag / s


def gradients(params, X, Y, rank, prop=None, M=1.0, biases=True):
    """(loss, pred, sparse gradients {name: array}, their magnitudes {name: array}, loss magnitude)."""
    P = len(X)
    u, i = X[:, 0], X[:, 1]
    pred, s, mag = forward(params, X, prop, M, biases)
    if rank == 1:
        b = P // 2
        x = pred[:b] - pred[b:]
        loss = float(np.logaddexp(0.0, -x).sum())
        sig = 1.0 / (1.0 + np.exp(x))
        dl = np.concatenate([-sig, sig])
        ddl = 0.25 * np.concatenate([mag[:b] + mag[b:]] * 2)     # |d dl| <= sigma' |d x|, sigma' <= 1/4
        loss_mag = float(np.logaddexp(0.0, -x).sum() + (mag[:b] + mag[b:]).sum())
    else:
        e = pred - np.asarray(Y, np.float64)
        loss = float((e * e).mean())
        dl = 2.0 * e / P
        ddl = 2.0 * (mag + np.abs(Y)) / P
        loss_mag = float(((e * e) + 2.0 * np.abs(e) * (mag + np.abs(Y))).sum() / P)
    r = dl / s
    r_abs = (np.abs(dl) + ddl) / s
    pu, qi = params['E_user'][u], params['E_item'][i]
    grads = {k: np.zeros_like(v) for k, v in params.items()}
    mags = {k: np.zeros_like(v) for k, v in params.items()}
    np.add.at(grads['E_user'], u, r[:, None] * qi)
    np.add.at(grads['E_item'], i, r[:, None] * pu)
    np.add.at(mags['E_user'], u, r_abs[:, None] * np.abs(qi))
    np.add.at(mags['E_item'], i, r_abs[:, None] * np.abs(pu))
    if biases:
        np.add.at(grads['user_bias'], u, r)
        np.add.at(grads['item_bias'], i, r)
        np.add.at(mags['user_bias'], u, r_abs)
        np.add.at(mags['item_bias'], i, r_abs)
        grads['global_bias'] = np.asarray(r.sum())
        mags['global_bias'] = np.asarray(r_abs.sum())
    return loss, pred, grads, mags, loss_mag


def pairs(params, X, Y, rank, prop=None, M=1.0):
    """Per-pair float64 terms of k_mf_step with tight first-order magnitudes (the `abs` of `gradients` bounds the
    sigmoid's slope by 1/4; here it is sigma (1 - sigma), so that a pair far in the tail is judged on its own scale):
    {'pred', 'scale', 'r' (the bias record d loss / d pred / scale), 'term' (the pair's loss term; 0 on the negative half
    of a BPR batch), 'gu' [P, D] = r q_i, 'gi' [P, D] = r p_u} and 'A_<name>' for each: |x_fp32 - x| <~ 2^-24 A_x."""
    P = len(X)
    u, i = X[:, 0], X[:, 1]
    pred, s, mag = forward(params, X, prop, M)
    A_pred = mag + np.abs(pred)
    if rank == 1:
        b = P // 2
        x = pred[:b] - pred[b:]
        A_x = A_pred[:b] + A_pred[b:] + np.abs(x)
        with np.errstate(over='ignore'):
            sig = 1.0 / (1.0 + np.exp(x))                        # sigmoid(-x)
        slope = sig * (1.0 - sig)
        dl = np.concatenate([-sig, sig])
        A_dl = np.concatenate([sig + slope * A_x] * 2)
        t = np.logaddexp(0.0, -x)
        term = np.concatenate([t, np.zeros(b)])
        A_term = np.concatenate([t + sig * A_x, np.zeros(b)])
    else:
        e = pred - np.asarray(Y, np.float64)
        A_e = A_pred + np.abs(np.asarray(Y, np.float64)) + np.abs(e)
        dl, A_dl = 2.0 * e / P, 2.0 * A_e / P
        term, A_term = e * e, 2.0 * np.abs(e) * A_e
    r = dl / s
    A_r = A_dl / s + np.abs(r)
    pu, qi = params['E_user'][u], params['E_item'][i]
    gu, gi = r[:, None] * qi, r[:, None] * pu
    return {'pred': pred, 'A_pred': A_pred, 'scale': s, 'r': r, 'A_r': A_r, 'term': term, 'A_term': A_term,
            'gu': gu, 'A_gu': A_r[:, None] * np.abs(qi) + np.abs(gu), 'gi': gi, 'A_gi': A_r[:, None] * np.abs(pu) + np.abs(gi)}


def apply_rule(p, st, gs, t, hp, kind):
    """One element-wise update of the runner's step; returns (new p, new state, g after l2 / clip / weight decay)."""
    g = np.clip(gs + 2.0 * hp['l2'] * p, -hp.get('clip', 50.0), hp.get('clip', 50.0)) + hp['weight_decay'] * p
    lr = hp['lr']
    if kind == 'adam':
        b1, b2, eps = hp.get('beta1', 0.9), hp.get('beta2', 0.999), hp.get('eps', 1e-8)
        m = b1 * st['m'] + (1 - b1) * g
        v = b2 * st['v'] + (1 - b2) * g * g
        denom = np.sqrt(v) / np.sqrt(1 - b2 ** t) + eps
        return p - lr / (1 - b1 ** t) * m / denom, {'m': m, 'v': v}, g
    if kind == 'adagrad':
        s = st['s'] + g * g
        return p - lr * g / (np.sqrt(s) + hp.get('eps', 1e-10)), {'s': s}, g
    return p - lr * g, {}, g


def step(params, state, t, X, Y, rank, hp, kind, prop=None, M=1.0, biases=True):
    """One training step at step count t.  Returns (params, state, loss, pred, info) with info = {'g': final gradients,
    'mag': their magnitudes (l2 / weight-decay terms included), 'loss_mag': magnitude of the loss}."""
    loss, pred, gs, mags, loss_mag = gradients(params, X, Y, rank, prop, M, biases)
    new_p, new_s, info = {}, {}, {'g': {}, 'mag': {}, 'loss_mag': loss_mag}
    for k, p in params.items():
        new_p[k], new_s[k], info['g'][k] = apply_rule(p, state[k], gs[k], t, hp, kind)
        info['mag'][k] = mags[k] + (2.0 * hp['l2'] + hp['weight_decay']) * np.abs(p)
    return new_p, new_s, loss, pred, info
