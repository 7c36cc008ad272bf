"""GPU check of the tensor-core training kernels (dccf_train_fwd_tc / dccf_train_bwd_tc) against the FP32 SIMT
kernels (dccf_score_fwd / dccf_bpr_bwd) stage by stage on the same inputs and the same random streams, plus
per-kernel timings.  Usage (on a B200): python tools/tc_train_check.py [--time]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dccf_b200 import kernels  # noqa: E402

D = 64


def rel(a, b):
    a, b = a.double(), b.double()
    den = float(b.abs().max())
    return float((a - b).abs().max()) / (den if den > 0 else 1.0)


def problem(seed, U, I, F, P, S, A):
    g = torch.Generator().manual_seed(seed)
    t = {'E_user': torch.randn(U, D, generator=g) * 0.05, 'E_item': torch.randn(I, D, generator=g) * 0.05,
         'W': torch.randn(D, D + F, generator=g) * 0.05, 'b': torch.randn(D, generator=g) * 0.05,
         'Feat': torch.randn(I, F, generator=g) / np.sqrt(F), 'expo': torch.rand(U, I, generator=g)}
    b = P // 2
    u = torch.randint(U, (b,), generator=g)
    X = torch.cat([torch.stack([u, torch.randint(I, (b,), generator=g)], 1),
                   torch.stack([u, torch.randint(I, (b,), generator=g)], 1)]).long()
    si = torch.randint(I, (P, S), generator=g).long()
    return {k: v.cuda().contiguous() for k, v in t.items()}, X.cuda(), si.cuda()


def run(path, t, X, si, F, S, A, rng, time_it=0):
    """path 'simt' | 'tc' -> dict of every intermediate and output of forward + backward."""
    U, I = t['E_user'].shape[0], t['E_item'].shape[0]
    P = X.shape[0]
    Z, K = S + 1, D + F
    N = P * Z * A
    dims = kernels.make_dims(U, I, F, S, A)
    expo = kernels.make_expo(dense=t['expo'])
    dev = X.device
    f32 = dict(dtype=torch.float32, device=dev)
    pred, ws_rows = torch.zeros(P, **f32), torch.zeros(N, **f32)
    save_h, save_w = torch.zeros(N, D, **f32), torch.zeros(P, Z, **f32)
    loss = torch.zeros(1, **f32)
    gu, gi = torch.zeros(P, D, **f32), torch.zeros(P * Z, D, **f32)
    ku, ki = torch.zeros(P, dtype=torch.int32, device=dev), torch.zeros(P * Z, dtype=torch.int32, device=dev)
    if path == 'simt':
        ns = kernels.bwd_splits(N)
        ws_wt = torch.zeros(K * D, **f32)
        fwd = lambda: kernels.score_fwd(dims, t['E_user'], t['E_item'], t['Feat'], t['W'], t['b'], expo, X, si, rng,
                                        pred, ws_rows, ws_wt, save_h, save_w, None)
    else:
        ns = kernels.train_bwd_splits(N, F)
        nk = kernels.train_fwd_ksplits(N, F)
        wimg = torch.zeros(kernels.train_w_image_floats(F), **f32)
        pre_part = torch.zeros(nk, N, D, **f32)
        dpre = torch.zeros(N, D, **f32)
        fwd = lambda: kernels.train_fwd_tc(dims, t['E_user'], t['E_item'], t['Feat'], t['W'], t['b'], expo, X, si, rng,
                                           pred, ws_rows, wimg, pre_part, save_h, save_w, None)
    gW_part, gb_part = torch.zeros(ns, D, K, **f32), torch.zeros(ns, D, **f32)
    if path == 'fused':
        terms = torch.zeros(P, **f32)

        def step():
            kernels.train_fwd_bwd_tc(dims, t['E_user'], t['E_item'], t['Feat'], t['W'], t['b'], expo, X, si, None, rng, 0,
                                     pred, loss, wimg, False, pre_part, dpre, terms, gW_part, gb_part, gu, gi, ku, ki,
                                     save_h, save_w, None, None, None)
        step()
        torch.cuda.synchronize()
        out = {'pred': pred, 'ws_rows': None, 'save_h': save_h, 'save_w': save_w, 'loss': loss, 'gW': gW_part.sum(0),
               'gb': gb_part.sum(0), 'gu': gu, 'gi': gi, 'ku': ku, 'ki': ki, 'splits': ns}
        if time_it:
            for _ in range(5):
                step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(time_it):
                step()
            e1.record()
            torch.cuda.synchronize()
            out['us_fwd'] = e0.elapsed_time(e1) * 1000.0 / time_it
            out['us_bwd'] = 0.0
        return out
    args = (dims, t['E_user'], t['E_item'], t['Feat'], t['W'], X, si, None, rng, 0, pred, save_h, save_w, loss, gW_part,
            gb_part, gu, gi, ku, ki)
    bwd = (lambda: kernels.bpr_bwd(*args)) if path == 'simt' else (lambda: kernels.train_bwd_tc(*args, dpre))
    fwd()
    bwd()
    torch.cuda.synchronize()
    out = {'pred': pred, 'ws_rows': ws_rows, 'save_h': save_h, 'save_w': save_w, 'loss': loss, 'gW': gW_part.sum(0),
           'gb': gb_part.sum(0), 'gu': gu, 'gi': gi, 'ku': ku, 'ki': ki, 'splits': ns}
    if time_it:
        for name, fn in (('fwd', fwd), ('bwd', bwd)):
            for _ in range(5):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(time_it):
                fn()
            e1.record()
            torch.cuda.synchronize()
            out['us_' + name] = e0.elapsed_time(e1) * 1000.0 / time_it
    return out


def compare(tag, a, b, tol):
    bad = []
    line = []
    # a pre-activation within 1e-7 of zero may pass the ReLU in one path and not in the other: the derivative of that
    # element then differs legitimately (a kink, not an error) — the gradient comparison is skipped for such runs
    flips = int(((a['save_h'] > 0) != (b['save_h'] > 0)).sum())
    for k in ('pred', 'ws_rows', 'save_h', 'save_w', 'loss', 'gW', 'gb', 'gu', 'gi'):
        if a[k] is None or b[k] is None:
            continue
        e = rel(b[k], a[k])
        line.append('%s %.2e' % (k, e))
        if flips and k in ('gW', 'gb', 'gi'):
            continue
        if not (e < tol.get(k, 2e-5)):
            bad.append(k)
    if flips:
        line.append('(%d ReLU gate flip(s): gW/gb/gi not compared)' % flips)
    for k in ('ku', 'ki'):
        if not torch.equal(a[k], b[k]):
            bad.append(k)
    print('%-44s %s  %s' % (tag, ' '.join(line), 'FAIL ' + ','.join(bad) if bad else 'ok'), flush=True)
    return not bad


def main():
    time_it = 200 if '--time' in sys.argv else 0
    ok = True
    torch.manual_seed(1234)        # explicit-noise runs are repeatable (a ReLU gate can flip on a 1e-7 difference)
    shapes = [(300, 500, 768, 256, 10, 2), (50, 70, 128, 38, 3, 1), (20, 30, 64, 2, 0, 1), (64, 64, 256, 130, 5, 3),
              (300, 500, 768, 64, 10, 2)]
    for (U, I, F, P, S, A) in shapes:
        t, X, si = problem(5, U, I, F, P, S, A)
        N = P * (S + 1) * A
        for mode in ('explicit', 'library', 'none'):
            if mode == 'explicit':
                noise = torch.randn(N, F, device='cuda') * 0.1
                mask = (torch.rand(N, D, device='cuda') < 0.8).float() / 0.8
                rng = kernels.make_rng(noise=noise, mask=mask, noise_std=0.1, p_drop=0.2)
            elif mode == 'library':
                rng = kernels.make_rng(noise_std=0.1, p_drop=0.2, seed=2019, offset=3, generate_noise=True,
                                       generate_mask=True)
            else:
                rng = kernels.make_rng()
            a = run('simt', t, X, si, F, S, A, rng)
            b = run('tc', t, X, si, F, S, A, rng)
            ok &= compare('U%d I%d F%d P%d S%d A%d %s' % (U, I, F, P, S, A, mode), a, b, {})
            c = run('fused', t, X, si, F, S, A, rng)
            ok &= compare('    fused', a, c, {})
    if time_it:
        U, I, F, P, S, A = 48000, 16000, 768, 256, 10, 2
        t, X, si = problem(7, U, I, F, P, S, A)
        rng = kernels.make_rng(noise_std=0.1, p_drop=0.2, seed=2019, offset=3, generate_noise=True, generate_mask=True)
        for path in ('simt', 'tc', 'fused'):
            o = run(path, t, X, si, F, S, A, rng, time_it=time_it)
            print('timing %-5s fwd %.1f us  bwd %.1f us  (back to back, no L2 flush; fwd incl. W prep + epilogue; '
                  'splits %d)' % (path, o['us_fwd'], o['us_bwd'], o['splits']), flush=True)
    print('ALL OK' if ok else 'MISMATCH', flush=True)
    return 0 if ok else 1


if __name__ == '__main__':
    sys.exit(main())
