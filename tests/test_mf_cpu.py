"""BiasedMF / IPSBiasedMF without a GPU: flags, main.py's class table, parameters and their initial values, the export
tool's block-by-block memmap, and the float64 MF trainer the GPU tests compare against — pinned to this repository's CPU
RecModel + torch optimizer step (itself pinned to the reference's runs by test_host_parity.py::
test_whole_run_equals_reference_run)."""
import argparse
import os
import sys

import numpy as np
import pytest
import torch

from mf_reference import init_state, step

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ips(tmp_path, U=7, I=11, seed=2019, M=0.1):
    from dccf_b200.models.IPSBiasedMF import IPSBiasedMF
    np.save(str(tmp_path / 'p.propensity.npy'), np.linspace(0.0, 1.0, I).astype(np.float32))
    return IPSBiasedMF(path=str(tmp_path), dataset='p', M=M, label_min=0, label_max=1, feature_num=0, user_num=U,
                       item_num=I, u_vector_size=64, i_vector_size=64, random_seed=seed,
                       model_path=str(tmp_path / 'm.pt'))


def test_flags_parse():
    from dccf_b200.models.BiasedMF import BiasedMF
    from dccf_b200.models.IPSBiasedMF import IPSBiasedMF
    a = IPSBiasedMF.parse_model_args(argparse.ArgumentParser(), 'IPSBiasedMF').parse_args([])
    assert a.M == 0.1 and a.u_vector_size == 64 and a.model_path == '../model/IPSBiasedMF/IPSBiasedMF.pt'
    assert IPSBiasedMF.parse_model_args(argparse.ArgumentParser()).parse_args(['--M', '0.25']).M == 0.25
    b = BiasedMF.parse_model_args(argparse.ArgumentParser(), 'BiasedMF').parse_args([])
    assert not hasattr(b, 'M') and b.model_path == '../model/BiasedMF/BiasedMF.pt'


def test_main_resolves_both_models():
    sys.path.insert(0, os.path.join(ROOT, 'src'))
    try:
        import main
    finally:
        sys.path.remove(os.path.join(ROOT, 'src'))
    from dccf_b200.models.BiasedMF import BiasedMF
    from dccf_b200.models.IPSBiasedMF import IPSBiasedMF
    assert main._resolve('BiasedMF') is BiasedMF and main._resolve('IPSBiasedMF') is IPSBiasedMF


def test_parameters_creation_order_and_initial_values(tmp_path):
    from dccf_b200.models.BaseModel import BaseModel
    U, I, seed = 7, 11, 2019
    model = _ips(tmp_path, U, I, seed)
    model.apply(model.init_paras)
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    assert shapes == {'uid_embeddings.weight': (U, 64), 'iid_embeddings.weight': (I, 64), 'user_bias.weight': (U, 1),
                      'item_bias.weight': (I, 1), 'global_bias': ()}
    assert [n for n, _ in model.named_children()] == ['uid_embeddings', 'iid_embeddings', 'user_bias', 'item_bias']
    # the same modules built by hand in the reference's order on the same seed, then N(0, 0.01) in module order
    torch.manual_seed(seed)
    mods = [torch.nn.Embedding(U, 64), torch.nn.Embedding(I, 64), torch.nn.Embedding(U, 1), torch.nn.Embedding(I, 1)]
    for m in mods:
        BaseModel.init_paras(m)
    for name, m in zip(('uid_embeddings', 'iid_embeddings', 'user_bias', 'item_bias'), mods):
        assert torch.equal(getattr(model, name).weight, m.weight), name
    assert model.global_bias.item() == pytest.approx(0.1) and model.global_bias.dtype == torch.float32
    assert model.propensity.shape == (I,) and model.M == 0.1
    with pytest.raises(RuntimeError, match='CUDA only'):
        model.predict({'X': torch.zeros((2, 2), dtype=torch.int64)})


def test_export_blocks_fill_the_memmap(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    try:
        import export_exposure
    finally:
        sys.path.remove(os.path.join(ROOT, 'tools'))
    full = np.random.RandomState(0).standard_normal((23, 9)).astype(np.float32)
    calls = []

    def compute(lo, hi):
        calls.append((lo, hi))
        return full[lo:hi]

    path = export_exposure.write_blocks(str(tmp_path / 'x.npy'), 23, 9, 5, compute)
    assert calls == [(0, 5), (5, 10), (10, 15), (15, 20), (20, 23)]
    got = np.load(path)
    assert got.dtype == np.float32 and np.array_equal(got, full)
    with pytest.raises(ValueError):
        export_exposure.write_blocks(str(tmp_path / 'y.npy'), 3, 3, 0, compute)


@pytest.mark.parametrize('kind', ['adam', 'gd', 'adagrad'])
@pytest.mark.parametrize('rank', [1, 0])
def test_reference_trainer_equals_recmodel_torch_step(kind, rank):
    """Without biases and fed the same batches, the float64 trainer follows the CPU RecModel trained by the runner's
    own step (loss + l2 * model.l2(), backward, clip_grad_value_(50), torch optimizer with weight_decay = l2)."""
    from dccf_b200.models.RecModel import RecModel
    from dccf_b200.runners.BaseRunner import BaseRunner
    U, I, P, steps, lr, l2 = 13, 17, 24, 4, 0.05, 1e-3
    model = RecModel(label_min=0, label_max=1, feature_num=0, user_num=U, item_num=I, u_vector_size=64,
                     i_vector_size=64, random_seed=5, model_path='unused.pt')
    model.apply(model.init_paras)
    with torch.no_grad():           # away from the init scale so that the loss terms are not all alike
        for p_ in model.parameters():
            p_.mul_(30.0)
    params = {'E_user': model.uid_embeddings.weight.detach().double().numpy().copy(),
              'E_item': model.iid_embeddings.weight.detach().double().numpy().copy()}
    state = init_state(params, kind)
    runner = BaseRunner(optimizer={'adam': 'Adam', 'gd': 'GD', 'adagrad': 'Adagrad'}[kind], learning_rate=lr, l2=l2)
    runner.show_progress = False
    model.optimizer = runner._build_optimizer(model)
    rs = np.random.RandomState(3)
    hp = {'lr': lr, 'l2': l2, 'weight_decay': l2}
    for t in range(1, steps + 1):
        X = np.stack([rs.randint(0, U, P), rs.randint(0, I, P)], 1).astype(np.int64)
        if rank == 1:
            X[P // 2:, 0] = X[:P // 2, 0]
        Y = rs.randint(1, 6, P).astype(np.float32) if rank == 0 else np.r_[np.ones(P // 2), np.zeros(P // 2)]
        batch = {'X': torch.from_numpy(X), 'Y': torch.from_numpy(Y.astype(np.float32)), 'rank': rank,
                 'dropout': 0.0, 'train': True}
        model.train()
        out = runner._fit_remaining(model, [batch], False, P, 0, None)
        params, state, loss, pred, _ = step(params, state, t, X, Y, rank, hp, kind, biases=False)
        assert float(out['loss']) == pytest.approx(loss, rel=2e-5)
        for k, mod in (('E_user', model.uid_embeddings), ('E_item', model.iid_embeddings)):
            got = mod.weight.detach().double().numpy()
            assert np.abs(got - params[k]).max() <= 2e-6 * np.abs(params[k]).max(), (t, k)
