"""Write the exposure inputs of DCCF from a trained IPSBiasedMF checkpoint (README.md:27-29 of the reference: the
exposure matrix is the U x I prediction of IPSBiasedMF):

    <path>/<dataset>/<dataset>.ips_expo_prob.npy   float32 [U, I]   (what DCCF loads by default)
    <path>/<dataset>/<dataset>.ipsmf.npz           the factors       (DCCF(expo_factors=...): exposure on the fly)

    python tools/export_exposure.py --path ../datasets/ --dataset Electronics --model_path ../model/IPSBiasedMF/x.pt

The matrix is computed on the GPU (full_catalogue.ipsmf_exposure, the tcgen05 GEMM) one block of users at a time and
written into a memory-mapped .npy, so host memory holds one block, not the whole matrix."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def write_blocks(path, n_users, n_items, block_users, compute):
    """Create the float32 [n_users, n_items] .npy at `path` and fill it with compute(lo, hi) -> [hi - lo, n_items]
    arrays, block by block."""
    if block_users <= 0:
        raise ValueError('--block_users must be positive, got %d' % block_users)
    out = np.lib.format.open_memmap(path, mode='w+', dtype=np.float32, shape=(n_users, n_items))
    for lo in range(0, n_users, block_users):
        hi = min(n_users, lo + block_users)
        out[lo:hi] = compute(lo, hi)
    out.flush()
    del out
    return path


def load_factors(model_path, propensity, M):
    """The make_ipsmf_factors dict (numpy) of an IPSBiasedMF checkpoint (the reference's state-dict keys)."""
    import torch
    sd = torch.load(model_path, map_location='cpu')
    prop = np.asarray(propensity, dtype=np.float32)
    if prop.shape != (sd['iid_embeddings.weight'].shape[0],):
        raise ValueError('propensity has shape %s, the checkpoint has %d items'
                         % (prop.shape, sd['iid_embeddings.weight'].shape[0]))
    f32 = lambda t: t.detach().to(torch.float32).contiguous().numpy()     # noqa: E731
    return {'mf_user': f32(sd['uid_embeddings.weight']), 'mf_item': f32(sd['iid_embeddings.weight']),
            'mf_user_bias': f32(sd['user_bias.weight']).reshape(-1), 'mf_item_bias': f32(sd['item_bias.weight']).reshape(-1),
            'mf_global_bias': np.float32(sd['global_bias'].item()), 'propensity': prop,
            'mf_min_propensity': np.float32(M)}


def export(path, dataset, model_path, M=0.1, block_users=4096):
    """Write both files; returns (matrix path, factors path)."""
    import torch
    from dccf_b200 import full_catalogue
    from dccf_b200.utils import global_p
    d = os.path.join(path, dataset)
    fac = load_factors(model_path, np.load(os.path.join(d, dataset + global_p.PROPENSITY_SUFFIX)), M)
    dev = {k: (torch.from_numpy(v).cuda() if v.ndim else float(v)) for k, v in fac.items()}
    U, I = fac['mf_user'].shape[0], fac['mf_item'].shape[0]

    def block(lo, hi):
        sub = dict(dev, mf_user=dev['mf_user'][lo:hi], mf_user_bias=dev['mf_user_bias'][lo:hi])
        return full_catalogue.ipsmf_exposure(sub).cpu().numpy()

    mat = write_blocks(os.path.join(d, dataset + '.ips_expo_prob.npy'), U, I, block_users, block)
    npz = os.path.join(d, dataset + '.ipsmf.npz')
    np.savez(npz, **fac)
    return mat, npz


def main(argv=None):
    ap = argparse.ArgumentParser(description='write <dataset>.ips_expo_prob.npy and <dataset>.ipsmf.npz from an '
                                             'IPSBiasedMF checkpoint')
    ap.add_argument('--path', default='../datasets/', help='data directory (as main.py --path)')
    ap.add_argument('--dataset', required=True)
    ap.add_argument('--model_path', required=True, help='IPSBiasedMF checkpoint (.pt state dict)')
    ap.add_argument('--M', type=float, default=0.1, help='propensity clamp the model was trained with')
    ap.add_argument('--block_users', type=int, default=4096, help='users per GPU block of the matrix')
    a = ap.parse_args(argv)
    for p in export(a.path, a.dataset, a.model_path, a.M, a.block_users):
        print(p)


if __name__ == '__main__':
    main()
