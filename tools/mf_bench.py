"""IPSBiasedMF training step and exposure export on one GPU -> profiles/mf_bench.json.

* Step: Electronics preset shape (48 000 users x 16 000 items, D = 64), Adam, --batch_size 128 (256 BPR pairs), random
  batches.  Per-step time by CUDA events around the graph replay (IPSBiasedMF.train_step), (a) with the 126 MB L2
  overwritten before every timed step and (b) back to back; train samples/s = 128 / back-to-back step time.
* The same model and loop run eagerly in torch (embedding lookups, BPR loss, l2 over all parameters, backward,
  clip_grad_value_(50), torch.optim.Adam with weight_decay) in the same process, for comparison.
* Export: full_catalogue.ipsmf_exposure of the whole U x I matrix for the Electronics and Yelp shapes, device time.
The card name and power limit are read in the same run and stored with the numbers.

    python tools/mf_bench.py [--steps 200] [--out profiles/mf_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in q.split(',')]
        return {'gpu': name, 'power_limit': limit}
    except Exception as e:          # the measurement stands without it, but says so
        return {'gpu': torch.cuda.get_device_name(0), 'power_limit': 'unknown (%s)' % e}


def timed(fn, n, flush=None):
    """Median and mean ms of fn() over n calls, each between two events; flush() (untimed) before each when given."""
    times = []
    for _ in range(n):
        if flush is not None:
            flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.mean(times))


def back_to_back(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--out', default=os.path.join('profiles', 'mf_bench.json'))
    a = ap.parse_args(argv)
    from dccf_b200 import full_catalogue, synth
    from dccf_b200.models.IPSBiasedMF import IPSBiasedMF
    assert torch.cuda.is_available(), 'the benchmark needs a CUDA device'
    dev = torch.device('cuda', 0)
    U, I, _ = synth.PRESETS['electronics']
    P = 256
    rs = np.random.RandomState(0)
    prop = rs.random_sample(I).astype(np.float32)
    model = IPSBiasedMF(path='', dataset='', M=0.1, label_min=0, label_max=1, feature_num=0, user_num=U, item_num=I,
                        u_vector_size=64, i_vector_size=64, random_seed=2019, model_path='/tmp/mf_bench.pt',
                        propensity=prop)
    model.apply(model.init_paras)
    model = model.cuda()
    model.optimizer = model.make_fused_optimizer(lr=1e-3, l2=1e-4)
    n_batches = 64
    Xs = []
    for _ in range(n_batches):
        X = np.stack([rs.randint(0, U, P), rs.randint(0, I, P)], 1).astype(np.int64)
        X[P // 2:, 0] = X[:P // 2, 0]
        Xs.append(torch.from_numpy(X).to(dev))
    Y = torch.cat([torch.ones(P // 2), torch.zeros(P // 2)]).to(dev)
    k = [0]

    def mf_step():
        model.train_step({'X': Xs[k[0] % n_batches], 'Y': Y, 'rank': 1})
        k[0] += 1

    scratch = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def flush():
        scratch.fill_(k[0])

    for _ in range(20):                     # eager first step, capture, replays
        mf_step()
    torch.cuda.synchronize()
    flushed = timed(mf_step, a.steps, flush)
    b2b = back_to_back(mf_step, a.steps)

    # the same model and loop in eager torch (the reference's runner step on the GPU)
    torch.manual_seed(2019)
    eu = torch.nn.Embedding(U, 64).to(dev)
    ei = torch.nn.Embedding(I, 64).to(dev)
    bu = torch.nn.Embedding(U, 1).to(dev)
    bi = torch.nn.Embedding(I, 1).to(dev)
    g = torch.nn.Parameter(torch.tensor(0.1, device=dev))
    params = list(eu.parameters()) + list(ei.parameters()) + list(bu.parameters()) + list(bi.parameters()) + [g]
    for p in params[:-1]:
        torch.nn.init.normal_(p, 0.0, 0.01)
    opt = torch.optim.Adam(params, lr=1e-3, weight_decay=1e-4)
    prop_d = torch.from_numpy(prop).to(dev)

    def torch_step():
        X = Xs[k[0] % n_batches]
        k[0] += 1
        opt.zero_grad()
        u, i = X[:, 0], X[:, 1]
        pred = ((eu(u) * ei(i)).sum(1) + bu(u).view(-1) + bi(i).view(-1) + g) / torch.clamp(prop_d[i], min=0.1)
        loss = -(pred[:P // 2] - pred[P // 2:]).sigmoid().log().sum()
        loss = loss + sum((p ** 2).sum() for p in params) * 1e-4
        loss.backward()
        torch.nn.utils.clip_grad_value_(params, 50)
        opt.step()

    for _ in range(20):
        torch_step()
    torch.cuda.synchronize()
    t_flushed = timed(torch_step, max(20, a.steps // 4), flush)
    t_b2b = back_to_back(torch_step, max(20, a.steps // 4))

    export = {}
    for name in ('electronics', 'yelp'):
        U2, I2, _ = synth.PRESETS[name]
        f = synth.make_ipsmf_factors(U2, I2)
        fd = {kk: (torch.from_numpy(v).to(dev) if v.ndim else float(v)) for kk, v in f.items()}
        full_catalogue.ipsmf_exposure(fd)
        torch.cuda.synchronize()
        export[name] = {'users': U2, 'items': I2,
                        'ms_median': timed(lambda: full_catalogue.ipsmf_exposure(fd), 10)[0]}
        del fd

    res = dict(gpu_info(), shape={'users': U, 'items': I, 'dim': 64, 'batch_size': 128, 'pairs': P, 'optimizer': 'Adam'},
               mf_step_us={'l2_flushed_median': 1e3 * flushed[0], 'back_to_back': 1e3 * b2b},
               train_samples_per_s=128 / (b2b * 1e-3),
               torch_eager_step_us={'l2_flushed_median': 1e3 * t_flushed[0], 'back_to_back': 1e3 * t_b2b},
               speedup_back_to_back=t_b2b / b2b, export_ms=export,
               adam_bytes_per_step=(U + I) * 64 * 24, steps=a.steps)
    os.makedirs(os.path.dirname(a.out) or '.', exist_ok=True)
    with open(a.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
