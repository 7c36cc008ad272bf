"""GD and Adagrad of the fused step, without a GPU: the numpy reference steps against torch.optim.SGD / Adagrad, the
runner's routing of --optimizer, and the rule field of the C ABI.

The reference steps below are what tests/test_gpu_optimizers.py compares the kernels with.  They extend
oracle/dccf_oracle.py (whose adam_step / train_step they mirror) to the reference's other two optimizers."""
import ctypes
import logging

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import dccf_oracle as O


# ------------------------------------------------------------------------------------------------
# loss += l2*sum p^2 ; clip_grad_value_(50) ; SGD / Adagrad(weight_decay=l2).step()
# (src/runners/BaseRunner.py:83-107,181,185,187; torch 2.11 optim/sgd.py, momentum 0, and optim/adagrad.py,
# lr_decay 0, initial_accumulator_value 0)
# ------------------------------------------------------------------------------------------------
def _grad(p, g_data, l2, weight_decay, clip, f):
    g = g_data.astype(f) + f(2.0 * l2) * p
    if clip > 0:
        g = np.clip(g, f(-clip), f(clip))
    return g + f(weight_decay) * p


def sgd_step(p, g_data, lr=1e-3, l2=1e-4, weight_decay=1e-4, clip=50.0, dtype=np.float32):
    f = dtype
    p = p.astype(f)
    g = _grad(p, g_data, l2, weight_decay, clip, f)
    return (p - f(lr) * g).astype(f)


def adagrad_step(p, g_data, s, lr=1e-3, l2=1e-4, weight_decay=1e-4, eps=1e-10, clip=50.0, dtype=np.float32):
    """Returns (p, state_sum)."""
    f = dtype
    p = p.astype(f)
    g = _grad(p, g_data, l2, weight_decay, clip, f)
    s = s.astype(f) + g * g
    p = p + f(-lr) * (g / (np.sqrt(s) + f(eps)))
    return p.astype(f), s.astype(f)


def train_step(params, state, t, X, sample_item, noise, mask, A, hp, loss_mode=0, Y=None, grad_dtype=np.float64,
               dtype=np.float32, optimizer='adam'):
    """oracle.dccf_oracle.train_step with the optimizer as a keyword: 'adam' (state m / v, the oracle's own step),
    'gd' (no state) or 'adagrad' (state 's').  Returns (new_params, new_state, loss, pred)."""
    if optimizer == 'adam':
        return O.train_step(params, state, t, X, sample_item, noise, mask, A, hp, loss_mode=loss_mode, Y=Y,
                            grad_dtype=grad_dtype, dtype=dtype)
    fwd = O.predict(params, X, sample_item, noise, mask, A, dtype=grad_dtype)
    loss = O.loss_bpr(fwd['pred']) if loss_mode == 0 else O.loss_mse(fwd['pred'], Y)
    grads = O.backward(params, X, sample_item, noise, mask, A, fwd, loss_mode=loss_mode, Y=Y, dtype=grad_dtype)
    new_params, new_state = dict(params), {}
    for k in ('E_user', 'E_item', 'W', 'b'):
        if optimizer == 'gd':
            new_params[k] = sgd_step(params[k], grads[k], dtype=dtype, **hp)
            new_state[k] = {}
        elif optimizer == 'adagrad':
            new_params[k], s = adagrad_step(params[k], grads[k], state[k]['s'], dtype=dtype, **hp)
            new_state[k] = {'s': s}
        else:
            raise ValueError(optimizer)
    return new_params, new_state, loss, fwd['pred']


# ------------------------------------------------------------------------------------------------
# 1. the reference steps against torch on the CPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['gd', 'adagrad'])
def test_reference_steps_equal_torch_optimizers(kind):
    """Five steps of loss = <c_t, p> + l2 * sum p^2, backward, clip_grad_value_(50), SGD / Adagrad(weight_decay=l2)
    step, in float32: the numpy steps follow torch within 1e-6.  Some data gradients are beyond +-50, so the clip bites."""
    rs = np.random.RandomState(4)
    lr, l2 = 1e-2, 1e-4
    shapes = {'E': (9, 64), 'W': (64, 80), 'b': (64,)}
    init = {k: (rs.standard_normal(s) * 0.05).astype(np.float32) for k, s in shapes.items()}
    coef = []
    for _ in range(5):
        c = {k: (rs.standard_normal(s) * 0.5).astype(np.float32) for k, s in shapes.items()}
        c['E'][0, :8] = 120.0            # clipped
        c['W'][3, :5] = -75.0            # clipped
        c['b'][:4] = 0.0                 # l2 / weight-decay terms only
        coef.append(c)
    ps = {k: torch.nn.Parameter(torch.from_numpy(v.copy())) for k, v in init.items()}
    params = list(ps.values())
    opt = torch.optim.SGD(params, lr=lr, weight_decay=l2) if kind == 'gd' else \
        torch.optim.Adagrad(params, lr=lr, weight_decay=l2)
    ref = {k: v.copy() for k, v in init.items()}
    sums = {k: np.zeros_like(v) for k, v in init.items()}
    for c in coef:
        opt.zero_grad()
        loss = sum((torch.from_numpy(c[k]) * p).sum() for k, p in ps.items()) + l2 * sum((p ** 2).sum() for p in params)
        loss.backward()
        torch.nn.utils.clip_grad_value_(params, 50)
        opt.step()
        for k in ref:
            if kind == 'gd':
                ref[k] = sgd_step(ref[k], c[k], lr=lr, l2=l2, weight_decay=l2)
            else:
                ref[k], sums[k] = adagrad_step(ref[k], c[k], sums[k], lr=lr, l2=l2, weight_decay=l2)
        for k, p in ps.items():
            assert rel_err(ref[k], p.detach().numpy()) < 1e-6, k
            if kind == 'adagrad':
                assert rel_err(sums[k], opt.state[p]['sum'].numpy()) < 1e-6, k


def test_train_step_default_is_the_oracle_adam_step():
    rs = np.random.RandomState(2)
    U, I, F, P, S, A = 6, 9, 16, 4, 2, 1
    params = {'E_user': (rs.standard_normal((U, 64)) * 0.05).astype(np.float32),
              'E_item': (rs.standard_normal((I, 64)) * 0.05).astype(np.float32),
              'W': (rs.standard_normal((64, 64 + F)) * 0.05).astype(np.float32),
              'b': (rs.standard_normal(64) * 0.05).astype(np.float32),
              'Feat': (rs.standard_normal((I, F)) / 4).astype(np.float32),
              'expo': rs.random_sample((U, I)).astype(np.float32)}
    X = np.stack([rs.randint(0, U, P), rs.randint(0, I, P)], 1).astype(np.int64)
    si = rs.randint(0, I, (P, S)).astype(np.int64)
    state = {k: {'m': np.zeros_like(params[k]), 'v': np.zeros_like(params[k])} for k in ('E_user', 'E_item', 'W', 'b')}
    hp = dict(lr=1e-3, l2=1e-4, weight_decay=1e-4)
    a = train_step(params, state, 1, X, si, None, None, A, hp)
    b = O.train_step(params, state, 1, X, si, None, None, A, hp)
    for k in ('E_user', 'E_item', 'W', 'b'):
        assert np.array_equal(a[0][k], b[0][k]) and np.array_equal(a[1][k]['v'], b[1][k]['v'])
    g = train_step(params, None, 1, X, si, None, None, A, hp, optimizer='gd')
    assert not np.array_equal(g[0]['W'], params['W']) and g[2] == b[2]


# ------------------------------------------------------------------------------------------------
# 2. --optimizer routing in the runner
# ------------------------------------------------------------------------------------------------
class _Fused(object):
    pass


class _FusedModel(torch.nn.Module):
    """A model with the fused step: make_fused_optimizer takes the optimizer kind."""

    def __init__(self):
        super(_FusedModel, self).__init__()
        self.w = torch.nn.Parameter(torch.zeros(3))
        self.calls = []

    def make_fused_optimizer(self, lr, l2, weight_decay=None, kind='adam'):
        self.calls.append(dict(lr=lr, l2=l2, weight_decay=weight_decay, kind=kind))
        return _Fused()


class _AdamOnlyModel(torch.nn.Module):
    """The signature the Adam call has always used: (lr, l2, weight_decay=None) and nothing else."""

    def __init__(self):
        super(_AdamOnlyModel, self).__init__()
        self.w = torch.nn.Parameter(torch.zeros(3))
        self.calls = []

    def make_fused_optimizer(self, lr, l2, weight_decay=None):
        self.calls.append(dict(lr=lr, l2=l2, weight_decay=weight_decay))
        return _Fused()


class _PlainModel(torch.nn.Module):
    def __init__(self):
        super(_PlainModel, self).__init__()
        self.w = torch.nn.Parameter(torch.zeros(3))


@pytest.mark.parametrize('name,kind', [('GD', 'gd'), ('Adagrad', 'adagrad')])
def test_runner_routes_gd_and_adagrad_to_the_fused_optimizer(name, kind, caplog):
    from dccf_b200.runners.BaseRunner import BaseRunner
    model = _FusedModel()
    with caplog.at_level(logging.INFO):
        opt = BaseRunner(optimizer=name, learning_rate=0.05, l2=3e-4)._build_optimizer(model)
    assert isinstance(opt, _Fused)
    assert model.calls == [dict(lr=0.05, l2=3e-4, weight_decay=3e-4, kind=kind)]
    assert 'Optimizer: ' + name in caplog.text


@pytest.mark.parametrize('name,cls', [('GD', torch.optim.SGD), ('Adagrad', torch.optim.Adagrad),
                                      ('Adam', torch.optim.Adam)])
def test_runner_keeps_torch_optimizers_for_models_without_the_fused_step(name, cls, caplog):
    from dccf_b200.runners.BaseRunner import BaseRunner
    with caplog.at_level(logging.INFO):
        opt = BaseRunner(optimizer=name, learning_rate=0.05, l2=3e-4)._build_optimizer(_PlainModel())
    assert type(opt) is cls
    assert opt.param_groups[0]['lr'] == 0.05 and opt.param_groups[0]['weight_decay'] == 3e-4
    assert 'Optimizer: ' + name in caplog.text


def test_runner_adam_call_is_unchanged():
    from dccf_b200.runners.BaseRunner import BaseRunner
    model = _AdamOnlyModel()
    opt = BaseRunner(optimizer='Adam', learning_rate=0.05, l2=3e-4)._build_optimizer(model)
    assert isinstance(opt, _Fused)
    assert model.calls == [dict(lr=0.05, l2=3e-4, weight_decay=3e-4)]


# ------------------------------------------------------------------------------------------------
# 3. the rule field of the C ABI
# ------------------------------------------------------------------------------------------------
def test_adam_struct_carries_the_rule_in_the_old_padding():
    """dccf_adam keeps its size and layout: `rule` sits where the padding after `step` was, so a zero-initialised
    struct still means Adam."""
    from dccf_b200 import _lib, kernels
    assert ctypes.sizeof(_lib.Adam) == 7 * 8 + 4 + 4 + 8
    assert _lib.Adam.rule.offset == _lib.Adam.step.offset + 4 == 60
    assert _lib.Adam().rule == 0 and kernels.make_adam(1e-3, 1e-4, 1e-4).rule == kernels.RULE_ADAM
    assert (kernels.RULE_ADAM, kernels.RULE_GD, kernels.RULE_ADAGRAD) == (0, 1, 2)
    assert kernels.make_adam(1e-3, 1e-4, 1e-4, rule=kernels.RULE_ADAGRAD).rule == 2


def test_adam_only_entry_points_reject_other_rules():
    """dccf_adam_sweep / _sweep_seg / _dense implement Adam only; an unknown rule is refused by every entry point.
    (Argument checks run before any device work, so this needs no GPU.)"""
    from dccf_b200 import _lib, kernels
    lib = _lib.load()
    for rule in (1, 2):
        hp = kernels.make_adam(1e-3, 1e-4, 1e-4, rule=rule)
        assert lib.dccf_adam_sweep(None, None, None, 0, None, None, 0, None, None, ctypes.byref(hp), None) == -1
        assert 'Adam only' in lib.dccf_last_error().decode()
        assert lib.dccf_adam_sweep_seg(None, None, None, 0, None, None, 0, 0, 0, 0, None, None, ctypes.byref(hp),
                                       None) == -1
        assert lib.dccf_adam_dense(None, None, None, 0, None, 0, 0, ctypes.byref(hp), None) == -1
        assert 'Adam only' in lib.dccf_last_error().decode()
    hp = kernels.make_adam(1e-3, 1e-4, 1e-4, rule=3)
    assert lib.dccf_adam_step(None, 0, None, 0, ctypes.byref(hp), None) == -1
    assert 'unknown optimizer rule' in lib.dccf_last_error().decode()
