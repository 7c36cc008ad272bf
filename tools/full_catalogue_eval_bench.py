"""Full-catalogue evaluation at the Yelp shape (BASELINE.json config 4): what known-item exclusion costs the fused
top-k, what the metrics kernel costs, and the rate of a whole evaluation pass.

    python tools/full_catalogue_eval_bench.py [--users 32000 --items 38000 --per_user 49 --iters 20] [--out FILE]

Synthetic histories from dccf_b200.synth.make_interactions (train / validation / test = 70 / 10 / 20 % of 49 items per
user), IPSBiasedMF factors from synth.make_ipsmf_factors.  Arms, alternated within every iteration, CUDA events, L2
flushed (256 MB overwritten) before every timed call:
  topk_k{K}          dccf_full_scores, fused top-K, no exclusion (item-side prep + GEMM + merge)
  topk_excl_k{K}     the same with each user's training + validation items excluded
  metrics_k{K}       dccf_topk_metrics on the excluded lists against the test items
  eval_pass          evaluate_full_catalogue(ndcg, recall, precision @5 and @10) end to end, host CSR building included
                     (host clock around the call, which ends in a device synchronise)
Prints one JSON line (and writes it to --out) with the card name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402
import torch  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i',
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def stats(ms):
    ms = np.asarray(ms)
    return {'median_ms': float(np.median(ms)), 'min_ms': float(ms.min()), 'max_ms': float(ms.max()), 'n': int(ms.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--users', type=int, default=32000)
    ap.add_argument('--items', type=int, default=38000)
    ap.add_argument('--per_user', type=int, default=49)
    ap.add_argument('--ks', type=str, default='5,10')
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('full_catalogue_eval_bench needs a CUDA device')
    from dccf_b200 import full_catalogue as fc
    from dccf_b200 import kernels, synth
    dev = torch.device('cuda', torch.cuda.current_device())
    ks = [int(k) for k in a.ks.split(',')]

    inter = synth.make_interactions(a.users, a.items, a.per_user, seed=2019)
    frames = {n: pd.DataFrame({'uid': v[0], 'iid': v[1], 'label': v[2], 'time': v[3]}) for n, v in inter.items()}
    dl = types.SimpleNamespace(label='label', train_df=frames['train'], validation_df=frames['validation'],
                               test_df=frames['test'], train_user_his=fc._split_his(frames['train'], 'label'))
    fac = synth.make_ipsmf_factors(a.users, a.items, seed=2019)
    f = {k: (torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) else float(v)) for k, v in fac.items()}

    # the sets the pass builds, kept for the per-kernel arms: every user of the shape, in uid order
    users, excl, pos = fc.evaluation_sets(dl, 'test', a.items)
    u = torch.from_numpy(users).to(dev)
    sub = dict(f, mf_user=f['mf_user'][u].contiguous(), mf_user_bias=f['mf_user_bias'][u].contiguous())
    ex = fc._device_csr(excl, dev)
    po, pi = fc._device_csr(pos, dev)
    U = len(users)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def topk(k, exclude):
        return kernels.full_scores(sub['mf_user'], sub['mf_item'], sub['mf_user_bias'], sub['mf_item_bias'],
                                   fc._col_scale(sub), float(sub['mf_global_bias']), materialise=False, k=k,
                                   exclude=exclude)[2]

    ids = {k: topk(k, ex) for k in ks}
    sums = torch.empty((1, 5), dtype=torch.float64, device=dev)
    arms = {}
    for k in ks:
        arms['topk_k%d' % k] = lambda k=k: topk(k, None)
        arms['topk_excl_k%d' % k] = lambda k=k: topk(k, ex)
        arms['metrics_k%d' % k] = lambda k=k: kernels.topk_metrics(ids[k], po, pi, [k], out_sums=sums)
    metrics = ['ndcg@5', 'recall@5', 'precision@5', 'ndcg@10', 'recall@10', 'precision@10']
    arms['eval_pass'] = lambda: fc.evaluate_full_catalogue(f, dl, metrics)
    ms = {n: [] for n in arms}
    for i in range(a.warmup + a.iters):
        for n, fn in arms.items():
            flush.fill_(float(i))
            torch.cuda.synchronize()
            if n == 'eval_pass':
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                t = (time.perf_counter() - t0) * 1e3
            else:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                t = e0.elapsed_time(e1)
            if i >= a.warmup:
                ms[n].append(t)
    name, power = card()
    res = {n: stats(v) for n, v in ms.items()}
    line = {'metric': 'full_catalogue_eval_users_per_s', 'value': U / (res['eval_pass']['median_ms'] / 1e3),
            'unit': 'users/s', 'gpu': name, 'power_limit': power, 'l2_flushed': True,
            'config': {'users_evaluated': U, 'users': a.users, 'items': a.items, 'per_user': a.per_user, 'ks': ks,
                       'excluded_items_per_user': float(np.diff(excl[0]).mean()),
                       'positives_per_user': float(np.diff(pos[0]).mean()), 'eval_metrics': metrics},
            'arms': res,
            'exclusion_overhead': {'k%d' % k: res['topk_excl_k%d' % k]['median_ms'] / res['topk_k%d' % k]['median_ms'] - 1.0
                                   for k in ks}}
    print(json.dumps(line))
    if a.out:
        with open(a.out, 'w') as fh:
            fh.write(json.dumps(line, indent=1) + '\n')


if __name__ == '__main__':
    main()
