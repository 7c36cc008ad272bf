"""Time of one training step with each optimizer of the fused step (Adam, GD, Adagrad) at a bench.py shape, and of the
autograd + torch.optim.SGD / Adagrad loop those two optimizers ran on before they had a fused step.

    python tools/optimizer_step_bench.py [--preset electronics] [--steps 200] [--warmup 10] [--reps 2]

Fused arm: the graph-replayed, device-resident step bench.py times (DCCF.begin_resident_epoch: one CUDA-graph launch per
step), one model per optimizer, the three optimizers alternating within each repetition.  Autograd arm: per batch what
BaseRunner.fit did for a torch optimizer — zero_grad, the autograd forward (confounders drawn on the CPU generator),
loss + l2 * model.l2(), backward, clip_grad_value_(50), step.  Every step is bracketed by CUDA events with the L2
flushed (bench.L2Flusher) before it.  The whole set runs --reps times, to show the spread.  Prints one JSON line with
the device name and its power limit (read by a query only)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402

KINDS = ('adam', 'gd', 'adagrad')


def device_info():
    info = {'device': torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm',
                              '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=60).stdout
        power, clock = [x.strip() for x in out.strip().split(',')]
        info.update(power_limit_w=float(power), max_sm_clock_mhz=float(clock))
    except (OSError, ValueError, subprocess.SubprocessError):
        info.update(power_limit_w=None, max_sm_clock_mhz=None)
    return info


def stats(ms):
    us = np.asarray(ms) * 1e3
    return {'n': int(len(us)), 'median_us': round(float(np.median(us)), 2), 'mean_us': round(float(us.mean()), 2),
            'p10_us': round(float(np.percentile(us, 10)), 2), 'p90_us': round(float(np.percentile(us, 90)), 2)}


def fused_steps(model, X_dev, seed, warmup, flush):
    """Per-step ms of the device-resident epoch X_dev (CUDA events around each graph launch, L2 flushed before)."""
    n = X_dev.shape[0]
    torch.manual_seed(seed)
    si = torch.randint(model.item_num, size=(n, 2 * bench.BATCH, bench.S)).to(X_dev.device)
    step = model.begin_resident_epoch(X_dev, si, bench.DROPOUT)
    n_first = n - step.remaining()          # run kernel by kernel before the graph is captured
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    torch.cuda.synchronize()
    for i in range(n_first, n):
        flush()
        ev[i][0].record()
        step()
        ev[i][1].record()
    torch.cuda.synchronize()
    model.check_ids()
    return [ev[i][0].elapsed_time(ev[i][1]) for i in range(max(warmup, n_first), n)]


def autograd_steps(model, opt, X_dev, warmup, flush):
    """Per-step ms of the reference's loop (src/runners/BaseRunner.py:175-188) with a torch optimizer."""
    Y = torch.cat([torch.ones(bench.BATCH), torch.zeros(bench.BATCH)]).to(X_dev.device)
    model.train()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(X_dev.shape[0])]
    torch.cuda.synchronize()
    for i in range(X_dev.shape[0]):
        flush()
        ev[i][0].record()
        opt.zero_grad()
        out = model({'X': X_dev[i], 'Y': Y, 'rank': 1, 'train': True, 'dropout': bench.DROPOUT})
        loss = out['loss'] + model.l2() * bench.L2
        loss.backward()
        torch.nn.utils.clip_grad_value_(model.parameters(), 50)
        opt.step()
        ev[i][1].record()
    torch.cuda.synchronize()
    return [ev[i][0].elapsed_time(ev[i][1]) for i in range(warmup, X_dev.shape[0])]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--preset', default='electronics', choices=sorted(bench.PRESETS))
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--reps', type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('optimizer_step_bench needs a CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    U, I = bench.PRESETS[args.preset]
    n = args.warmup + args.steps
    X_dev = torch.from_numpy(bench.synth_batches(n, U, I, bench.SEED + 1)).to(dev)
    flush = bench.L2Flusher(dev)
    fused = {}
    for kind in KINDS:
        fused[kind] = bench.build_model(U, I, dev)
        fused[kind].optimizer = fused[kind].make_fused_optimizer(lr=bench.LR, l2=bench.L2, kind=kind)
    ref = {}
    for kind, cls in (('gd', torch.optim.SGD), ('adagrad', torch.optim.Adagrad)):
        m = bench.build_model(U, I, dev)
        ref[kind] = (m, cls(m.parameters(), lr=bench.LR, weight_decay=bench.L2))
    reps = []
    for rep in range(args.reps):
        r = {}
        for kind in KINDS:
            r['fused_' + kind] = stats(fused_steps(fused[kind], X_dev, bench.SEED + 20 + rep, args.warmup, flush))
        for kind in ('gd', 'adagrad'):
            r['autograd_' + kind] = stats(autograd_steps(ref[kind][0], ref[kind][1], X_dev, args.warmup, flush))
        reps.append(r)
    arms = list(reps[0])
    summary = {a: {'median_us': [rp[a]['median_us'] for rp in reps]} for a in arms}
    speedup = {k: round(float(np.median([rp['autograd_' + k]['median_us'] / rp['fused_' + k]['median_us']
                                         for rp in reps])), 1) for k in ('gd', 'adagrad')}
    out = dict(device_info(), tool='optimizer_step_bench', preset=args.preset, users=U, items=I,
               pairs_per_step=2 * bench.BATCH, steps=args.steps, warmup=args.warmup, l2_flushed=True,
               fused='graph-replayed device-resident step (begin_resident_epoch)',
               autograd='zero_grad + autograd forward + loss + l2 + backward + clip + torch.optim step',
               reps=reps, median_us_per_rep=summary, speedup_fused_over_autograd=speedup)
    print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
