"""Epoch time of rating prediction (--rank 0, MSE loss) through BaseRunner.fit with each optimizer of the fused step
(Adam, GD, Adagrad): the device-resident epoch against the step-by-step loop it replaces.

    python tools/rank0_fit_bench.py [--preset electronics] [--batches 4000] [--reps 3]

Workload: --batches batches of 128 rating pairs (bench.py's users, popularity-skewed items, labels uniform in [1, 5])
and a ragged last batch of 57 pairs, the model of bench.py.  Resident arm: `runner.fit` — the full batches run from
the device-resident epoch (one CUDA-graph launch per step, labels staged on the device), the ragged one step by step.
Step-by-step arm: `runner._fit_remaining` over the same batches, the schedule fit used for --rank 0 before: per step a
Python train_step, a host confounder draw and the copies into the graph's input buffers.  Both arms start from the same
weights and draw the same confounders (the CPU generator is re-seeded before every epoch), so their parameters must
end bit-identical; that is checked.  One warm-up epoch per arm (graph capture), then --reps epochs, the arms
alternating within each repetition.  Per arm: seconds per epoch (host clock, ending in a device synchronise) and us
per step (CUDA events around every step call, the L2 not flushed: steps run back to back as in training).  Prints one
JSON line with the device name and its power limit (read by a query only)."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from optimizer_step_bench import device_info, stats  # noqa: E402

KINDS = ('adam', 'gd', 'adagrad')
RUNNER_NAME = {'adam': 'Adam', 'gd': 'GD', 'adagrad': 'Adagrad'}
RAGGED = 57


class _Batches(object):
    """A --rank 0 data processor whose epoch is a fixed list of device batches."""
    rank = 0

    def __init__(self, batches):
        self.batches = batches

    def prepare_batches(self, data, batch_size, train):
        return [dict(b) for b in self.batches]


def rating_batches(n, U, I, seed, device):
    X = bench.synth_batches(n + 1, U, I, seed)[:, :bench.BATCH]          # [n + 1, 128, 2]: the positives' pairs
    Y = np.random.RandomState(seed + 1).uniform(1.0, 5.0, size=(n + 1, bench.BATCH)).astype(np.float32)
    out = [{'X': torch.from_numpy(X[k]).to(device), 'Y': torch.from_numpy(Y[k]).to(device), 'rank': 0}
           for k in range(n)]
    out.append({'X': torch.from_numpy(X[n, :RAGGED]).to(device), 'Y': torch.from_numpy(Y[n, :RAGGED]).to(device),
                'rank': 0})
    return out


def timed(model):
    """Record CUDA events around every training step the runner makes (train_step calls and resident-epoch steps)."""
    events = []

    def around(fn):
        def call(*a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **kw)
            e1.record()
            events.append((e0, e1))
            return out
        return call

    model.train_step = around(model.train_step)
    begin = model.begin_resident_epoch

    def begin_timed(*a, **kw):
        step = begin(*a, **kw)
        if step is None:
            return None
        wrapped = around(step)
        wrapped.remaining, wrapped.first = step.remaining, step.first
        return wrapped
    model.begin_resident_epoch = begin_timed
    return events


def epoch(runner, model, dp, resident, seed):
    """(seconds, per-step ms) of one epoch."""
    events = model.__dict__['_bench_events']
    del events[:]
    torch.manual_seed(seed)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if resident:
        runner.fit(model, None, dp, epoch=0)
    else:
        batches = runner.batches_add_control(dp.prepare_batches(None, runner.batch_size, train=True), train=True)
        model.train()
        runner._fit_remaining(model, batches, True, runner.batch_size, 0, None)
        model.eval()
        model.check_ids()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    return sec, [a.elapsed_time(b) for a, b in events]


def main():
    from dccf_b200.runners.BaseRunner import BaseRunner
    ap = argparse.ArgumentParser()
    ap.add_argument('--preset', default='electronics', choices=sorted(bench.PRESETS))
    ap.add_argument('--batches', type=int, default=4000)
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('rank0_fit_bench needs a CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    U, I = bench.PRESETS[args.preset]
    dp = _Batches(rating_batches(args.batches, U, I, bench.SEED + 1, dev))
    arms = {}
    for kind in KINDS:
        for resident in (True, False):
            model = bench.build_model(U, I, dev)
            model.optimizer = model.make_fused_optimizer(lr=bench.LR, l2=bench.L2, kind=kind)
            model.__dict__['_bench_events'] = timed(model)
            runner = BaseRunner(optimizer=RUNNER_NAME[kind], learning_rate=bench.LR, l2=bench.L2,
                                batch_size=bench.BATCH, dropout=bench.DROPOUT, metrics='rmse')
            runner.show_progress = False
            arms[(kind, resident)] = (runner, model)
    for (kind, resident), (runner, model) in arms.items():      # warm-up: graph capture, module loads
        epoch(runner, model, dp, resident, bench.SEED + 30)
    res = {(k, r): {'s_per_epoch': [], 'step_ms': []} for k, r in arms}
    for rep in range(args.reps):
        for kind in KINDS:
            for resident in (True, False):
                runner, model = arms[(kind, resident)]
                sec, ms = epoch(runner, model, dp, resident, bench.SEED + 40 + rep)
                res[(kind, resident)]['s_per_epoch'].append(round(sec, 4))
                res[(kind, resident)]['step_ms'] += ms
    out_arms, identical = {}, {}
    for kind in KINDS:
        for resident in (True, False):
            r = res[(kind, resident)]
            out_arms['%s_%s' % (kind, 'resident' if resident else 'step_by_step')] = dict(
                s_per_epoch=r['s_per_epoch'], steps_per_epoch=args.batches + 1, step_us=stats(r['step_ms']))
        a, b = arms[(kind, True)][1], arms[(kind, False)][1]
        identical[kind] = all(torch.equal(p, q) for p, q in zip(a.parameters(), b.parameters()))
    speedup = {k: round(float(np.median(res[(k, False)]['s_per_epoch']) / np.median(res[(k, True)]['s_per_epoch'])), 2)
               for k in KINDS}
    out = dict(device_info(), tool='rank0_fit_bench', preset=args.preset, users=U, items=I, task='--rank 0 (MSE)',
               pairs_per_step=bench.BATCH, full_batches=args.batches, ragged_batch=RAGGED, reps=args.reps,
               l2_flushed=False, resident='runner.fit (device-resident epoch + ragged batch step by step)',
               step_by_step='runner._fit_remaining over the same batches', arms=out_arms,
               epoch_speedup_resident=speedup, parameters_bit_identical=identical)
    print(json.dumps(out), flush=True)
    if not all(identical.values()):
        raise SystemExit('resident and step-by-step epochs ended with different parameters')


if __name__ == '__main__':
    main()
