"""bench.py — DCCF training (samples/s) and 1000-negative evaluation (users/s) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--preset electronics]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One JSON line on stdout (rank 0).  A "step" is one training batch of the reference configuration
(--batch_size 128 -> 256 scored pairs: 128 positives + their sampled negatives; S=10 confounders, A=2,
std 0.1, dropout 0.2, Adam lr 1e-3, l2 1e-4) on synthetic Electronics-shaped data (BASELINE.json configs[1]);
`value` is train samples/s with the batches already in HBM, `e2e` the same through the public API
(model.train_step) from pinned host buffers — ids staged and uploaded every step, confounders drawn on the torch
CPU generator every step, the loss copied back every step.  The `eval` object holds the evaluation half of the
metric: users/s for ranking each test user's positive against test_neg_n = 1000 sampled negatives (scoring +
on-device top-k/ndcg/recall/precision@5 in one ranker launch).

Further objects on the same line (tools/bench_legs.py):
  dp_parity            N > 1: the data-parallel step equals the single-GPU step on the concatenated batch (checked BEFORE
                       timing; the process exits with rc 3 when it does not) + replica checksum after the timed steps
  config3_cds          BASELINE.json configs[2]: the same train / eval pair at the CDs_and_Vinyl shape
  config4_full_catalogue  configs[3]: Yelp shape, full-catalogue tcgen05 GEMM + top-k, users sharded over the N ranks
  config5_scaled       configs[4]: 10 M x 1 M, row-sharded user table, on-the-fly IPSBiasedMF exposure
  eval_noise_free / eval_projected_noise / gpu_eager_reference / cpu_baseline   N = 1 only (child process for the first two)
--legs selects them (default: all that apply); --no-extra-legs / --no-cpu-baseline skip groups.
Every roofline object reports `frac` on ALGORITHMIC work (SURVEY.md §8d flops / bytes); `frac_issued` counts the three
TF32 products the tensor cores actually execute per FP32 product.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark leaves no __pycache__ in it

import numpy as np  # noqa: E402
import torch  # noqa: E402

PRESETS = {            # SURVEY.md §8d: (users, items) — the reference ships no data, shapes are ours
    'tiny': (2000, 5000),
    'electronics': (48000, 16000),
    'cds': (24000, 20000),
    'yelp': (32000, 38000),
}
D, F, S, A = 64, 768, 10, 2
Z, R = S + 1, (S + 1) * A
BATCH = 128
EVAL_BATCH = 16384
TEST_NEG_N = 1000
LR, L2, DROPOUT, STD = 1e-3, 1e-4, 0.2, 0.1
SEED = 2019

# algorithmic work per scored pair (SURVEY.md §8d)
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the step's kernels at the electronics shape, from ONE
# `ncu --set full --clock-control none` capture (cold cache before every kernel), see profiles/
NCU_TRAFFIC_SOURCE = 'profiles/r2_ncu_train_summary.csv (ncu --set full --clock-control none, mean per launch, cold cache)'
NCU_EVAL_TRAFFIC_BYTES = 8.779776e6        # k_row_scores_tc<2>, one 16384-pair batch: dram read (0 written)
NCU_EVAL_TRAFFIC_SOURCE = ('profiles/r2_ncu_eval_summary.csv (ncu --set full --clock-control none, one launch = one '
                           '16384-pair batch, cold cache)')
NCU_TRAFFIC_BYTES = {'k_train_fwd_tc': 1.88e6, 'k_train_mid': 6.05e6, 'k_train_bwd_tc': 2.91e6, 'k_adam_touched': 8.02e6,
                     'k_adam_untouched': 49.26e6 + 0.46e6, 'k_link_ids': 4.37e6}
# round 2 captures (per launch, cold cache, `ncu --set full --clock-control none`): dram__bytes_read.sum + dram__bytes_write.sum
NCU_R2 = {'source': 'profiles/r2_ncu_eval_summary.csv (ncu --set full --clock-control none, per launch, cold cache)',
          'k_gather_scores': 9.47e6,          # one 16384-pair batch (mean of three launches)
          'k_row_scores_tc_64': 8.40e6,       # one 16384-pair batch, 64-wide operand
          'k_confounder_draw': 1.0e4,         # one 163 840-id draw: nothing read, ids written through L2
          'k_rank_stream': 8.96e6,            # 1024 users x 1001 candidates: scores + labels once (8.2 MB algorithmic)
          'k_full_scores_topk': 30.27e6}      # Yelp shape, one GPU: user factors + the pre-split item images in, k ids out
                                              # (profiles/r2_ncu_full_catalogue_summary.csv)
FLOP_FWD_PAIR = R * (2 * (D + F) * D + 4 * D)
FLOP_BWD_PAIR = R * (2 * (D + F) * D + 2 * D * D + 2 * D)
BYTES_PAIR = 16 + 4 * D + 4 * D * Z + 4 * F + 4 * Z
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12


def measured_peaks():
    """(HBM GB/s, dense bf16 TFLOP/s burst, source)."""
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d['hbm_gbs']), float(d.get('bf16_tflops', 1590.0)), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 1590.0, 'fallback (B200_PROFILING.md)'


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    FIELDS = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._thread = None

    def _run(self):
        try:
            proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                                     '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                    stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        try:
            while not self._stop.is_set():
                line = proc.stdout.readline()
                if not line:
                    break
                self.samples.append([x.strip() for x in line.split(',')])
        finally:
            proc.terminate()

    def __enter__(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        time.sleep(0.15)
        self._stop.set()
        self._thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, s[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def synth_batches(n_steps, U, I, seed):
    """[n_steps, 2*BATCH, 2] int64: rows [0,128) positives, [128,256) their negatives, same user."""
    rs = np.random.RandomState(seed)
    pop = 1.0 / np.arange(1, I + 1, dtype=np.float64) ** 0.8
    cdf = np.cumsum(pop / pop.sum())
    u = rs.randint(0, U, size=(n_steps, BATCH))
    pos = np.minimum(np.searchsorted(cdf, rs.random_sample((n_steps, BATCH))), I - 1)
    neg = rs.randint(0, I, size=(n_steps, BATCH))
    X = np.empty((n_steps, 2 * BATCH, 2), dtype=np.int64)
    X[:, :BATCH, 0] = u
    X[:, BATCH:, 0] = u
    X[:, :BATCH, 1] = pos
    X[:, BATCH:, 1] = neg
    return X


def synth_eval_set(n_users, U, I, seed):
    """n_users test users x (1 positive + TEST_NEG_N sampled negatives): X [rows,2], uid, iid, Y."""
    rs = np.random.RandomState(seed + 1)
    users = rs.choice(U, n_users, replace=False)
    n_c = 1 + TEST_NEG_N
    uid = np.repeat(users, n_c)
    iid = np.empty((n_users, n_c), dtype=np.int64)
    for g in range(n_users):
        iid[g] = rs.choice(I, n_c, replace=False)
    Y = np.zeros((n_users, n_c), dtype=np.float32)
    Y[:, 0] = 1.0
    iid, Y = iid.reshape(-1), Y.reshape(-1)
    return np.stack([uid, iid], 1).astype(np.int64), uid, iid, Y


def build_model(U, I, device, std=STD):
    from dccf_b200.models.DCCF import DCCF
    g = torch.Generator(device='cpu').manual_seed(SEED + 5)
    feat = torch.randn((I, F), generator=g) / (F ** 0.5)
    gd = torch.Generator(device=device).manual_seed(SEED + 6)
    expo = torch.rand((U, I), generator=gd, device=device)              # "random ips_expo_prob" (BASELINE.json)
    torch.manual_seed(SEED)
    model = DCCF(path='', dataset='', sentence_model='', sample_num=S, attribute_num=A, std=std, label_min=0,
                 label_max=1, feature_num=0, user_num=U, item_num=I, u_vector_size=D, i_vector_size=D, n_layers=1,
                 random_seed=SEED, model_path='/tmp/dccf_bench.pt', feature_embedding=feat, expo_prob=expo)
    model.apply(model.init_paras)                                         # N(0, 0.01) random-init weights
    model = model.to(device)
    model.optimizer = model.make_fused_optimizer(lr=LR, l2=L2)
    return model


class L2Flusher(object):
    """Writes a 256 MiB buffer (> the 126 MB L2) between timed iterations."""

    def __init__(self, device):
        self.buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)
        self.v = 0.0

    def __call__(self):
        self.v += 1.0
        self.buf.fill_(self.v)


DUMP_ARRAY_BYTES = 16 * 2 ** 20     # per array: a dump has at most eight arrays, so it stays under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy: float64 where the path computes in float64, float32 otherwise.  An
    array larger than DUMP_ARRAY_BYTES keeps a fixed sample of its rows, as many as fit:
    np.sort(np.random.RandomState(SEED).choice(n_rows, n_kept, replace=False))."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > DUMP_ARRAY_BYTES:
            n_kept = DUMP_ARRAY_BYTES // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.RandomState(SEED).choice(a.shape[0], n_kept, replace=False))]
        np.save(os.path.join(out_dir, name + '.npy'), a)


def dist_max(x, world):
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device='cuda')
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def bench_train(model, X_all, steps, warmup, world, flush, keep_outputs=False):
    """Returns dict with device-resident timing (CUDA events per step, L2 flushed in between, max over ranks),
    per-stage times and the end-to-end timing from pinned host buffers.  keep_outputs: also 'outputs', what the last
    timed step returned (prediction, loss) and the parameters it left, as host arrays."""
    from dccf_b200 import kernels
    dev = next(model.parameters()).device
    n = warmup + steps
    Y = torch.cat([torch.ones(BATCH), torch.zeros(BATCH)]).to(dev)
    I = model.item_num

    # ---- value: the epoch's batches and confounder draws resident in HBM; every step is ONE CUDA-graph
    # launch that fetches its batch through a device-side cursor (DCCF.begin_resident_epoch) ----------------
    X_dev = torch.from_numpy(X_all[:n]).to(dev)
    torch.manual_seed(SEED + 11)
    si_dev = torch.randint(I, size=(n, 2 * BATCH, S)).to(dev)
    step = model.begin_resident_epoch(X_dev, si_dev, DROPOUT)
    n_first = n - step.remaining()              # steps already run kernel by kernel to load the modules
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(n)]
    launches0 = kernels.LAUNCHES[0]
    barrier(world)
    for i in range(n_first, n):
        if i == warmup:
            barrier(world)
            launches0 = kernels.LAUNCHES[0]
        flush()
        ev[i][0].record()
        out = step()
        ev[i][1].record()
    barrier(world)
    outputs = None
    if keep_outputs:            # before the back-to-back and end-to-end steps below train the model further
        outputs = {'train_prediction': out['prediction'], 'train_loss': out['loss']}
        outputs.update(('param_' + k.replace('.', '_'), p) for k, p in model.named_parameters())
        outputs = {k: v.detach().cpu().numpy() for k, v in outputs.items()}
    launches = kernels.LAUNCHES[0] - launches0
    per_step = [ev[i][0].elapsed_time(ev[i][1]) for i in range(max(warmup, n_first), n)]
    total_ms = dist_max(float(np.sum(per_step)) * steps / len(per_step), world)
    model.check_ids()

    # the same K steps back to back (no L2 flush, one event pair): the steady state of a real epoch, where
    # the 50 MB of parameters and Adam state stay L2-resident between steps — reported next to the value
    torch.manual_seed(SEED + 14)
    si_b2b = torch.randint(I, size=(steps, 2 * BATCH, S)).to(dev)
    step2 = model.begin_resident_epoch(X_dev[warmup:warmup + steps].contiguous(), si_b2b, DROPOUT)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    n_b2b = 0
    while step2.remaining() > 0:
        step2()
        n_b2b += 1
    e1.record()
    barrier(world)
    b2b_ms = dist_max(e0.elapsed_time(e1) / max(1, n_b2b), world)

    # ---- per-kernel times of the SAME captured step (extra replays of the same graph, L2 flushed before each
    # measured step exactly as in the timed loop): the kernels' own CTAs stamp %globaltimer at start / end
    # (dccf_b200/debug.py) — CUDA events cannot bracket the nodes of a graph.  Data-parallel runs (a different,
    # unfused step) fall back to CUDA events between the stages of a kernel-by-kernel step. --------------------
    kernels_us, timeline_step_us, stage_ms = {}, 0.0, None
    if model._split_step_ok(0, 2 * BATCH):
        from dccf_b200.debug import StepTimeline
        n_t = 30
        torch.manual_seed(SEED + 15)
        si_t = torch.randint(I, size=(3 * n_t, 2 * BATCH, S)).to(dev)
        X_t = X_dev[torch.arange(3 * n_t, device=dev) % n].contiguous()
        step3 = model.begin_resident_epoch(X_t, si_t, DROPOUT)
        with StepTimeline(dev) as tl:
            while step3.remaining() >= 3:
                step3()
                step3()                 # no host synchronisation before the measured step: it starts on a busy GPU
                flush()
                tl.arm()
                step3()
                tl.collect()
            kernels_us, timeline_step_us = tl.summary()
        if world > 1 and os.environ.get('DCCF_BENCH_RANK_TIMELINES'):
            # diagnostics: every rank's own timeline of the captured step (stderr), absolute globaltimer of the first kernel
            rank_ = int(os.environ.get('RANK', '0'))
            starts = [int(min(int(r[i, 0]) for i in range(r.shape[0]) if r[i, 1] != 0)) for r in tl.rows]
            print(json.dumps({'rank': rank_, 'step_us': timeline_step_us, 'first_kernel_ns_mod': [s_ % 10**9 for s_ in starts[:6]],
                              'kernels': {k_: [round(v_['start_us'], 1), round(v_['end_us'], 1)] for k_, v_ in kernels_us.items()}}),
                  file=sys.stderr, flush=True)
    else:
        n_s = min(n, warmup + 50)
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(n_s)]
        stage_ms = np.zeros(3)
        for i in range(n_s):
            flush()
            fd = {'X': X_dev[i], 'Y': Y, 'rank': 1, 'train': True, 'dropout': DROPOUT, 'sample_item': si_dev[i]}
            model.train_step(fd, stage_events=evs[i])
        barrier(world)
        for i in range(warmup, n_s):
            for st in range(3):
                stage_ms[st] += evs[i][st].elapsed_time(evs[i][st + 1])
        stage_ms /= max(1, n_s - warmup)

    # ---- e2e: the public API (model.train_step) fed from the host every step ------------------------------------
    # Per step: ids in pinned host memory -> staged with the step's confounder draw (torch CPU generator, DCCF.py:72)
    # and uploaded by one asynchronous copy, one CUDA-graph launch, the loss copied back into a pinned slot.  The
    # host does not wait for the device inside the loop (the reference's loop does not either: it reads the loss at
    # check_epoch, src/runners/BaseRunner.py:247-248); the timed region ends with a synchronise.  The L2 flush between
    # steps is kept (same kernels as `value`); its device time, measured by events around every flush, is subtracted.
    X_pin = torch.from_numpy(X_all[:n]).pin_memory()
    losses = torch.zeros(n, dtype=torch.float32).pin_memory()
    torch.manual_seed(SEED + 12)
    fl_ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(n)]

    def e2e_step(i):
        fl_ev[i][0].record()
        flush()
        fl_ev[i][1].record()
        out = model.train_step({'X': X_pin[i], 'Y': Y, 'rank': 1, 'train': True, 'dropout': DROPOUT})
        losses[i:i + 1].copy_(out['loss'].view(1), non_blocking=True)

    barrier(world)
    for i in range(warmup):
        e2e_step(i)
    barrier(world)
    t0 = time.perf_counter()
    for i in range(warmup, n):
        e2e_step(i)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    flush_s = sum(fl_ev[i][0].elapsed_time(fl_ev[i][1]) for i in range(warmup, n)) / 1e3
    e2e_s = dist_max(max(t1 - t0 - flush_s, 1e-9), world)
    loss = float(losses[n - 1])
    assert np.isfinite(losses.numpy()).all()
    # the same loop with the host waiting for every step's loss before it starts the next (latency-bound)
    n_sync = min(steps, 50)
    sync_s = 0.0
    for i in range(n_sync):
        flush()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = model.train_step({'X': X_pin[warmup + i], 'Y': Y, 'rank': 1, 'train': True, 'dropout': DROPOUT})
        float(out['loss'].item())
        sync_s += time.perf_counter() - t0
    sync_s = dist_max(sync_s / max(1, n_sync), world)
    return {'total_ms': total_ms, 'stage_ms': stage_ms, 'kernels_us': kernels_us, 'timeline_step_us': timeline_step_us,
            'launches': launches, 'e2e_s': e2e_s, 'e2e_sync_s_per_step': sync_s, 'b2b_ms': b2b_ms,
            'h2d': 2 * BATCH * 2 * 8 + 2 * BATCH * S * 8, 'd2h': 4, 'last_loss': loss, 'outputs': outputs}


def bench_eval(model, n_users, warm_batches, world, rank, flush, keep_outputs=False):
    """Scores n_users x 1001 candidates in eval batches of 16384 pairs and ranks them on the device.  keep_outputs:
    also 'outputs', the predictions and metrics of the last timed pass, as host arrays."""
    from dccf_b200.models.BaseModel import candidate_layout, rank_sums_device
    dev = next(model.parameters()).device
    U, I = model.user_num, model.item_num
    X, uid, iid, Y = synth_eval_set(n_users, U, I, SEED + 100 * rank)
    rows = X.shape[0]
    bounds = [(a, min(rows, a + EVAL_BATCH)) for a in range(0, rows, EVAL_BATCH)]
    cand, off = candidate_layout(uid)
    cand_d, off_d = (None if cand is None else torch.from_numpy(cand).to(dev)), torch.from_numpy(off).to(dev)
    Y_d, iid_d = torch.from_numpy(Y).to(dev), torch.from_numpy(iid).to(dev)
    X_d = torch.from_numpy(X).to(dev)
    torch.manual_seed(SEED + 13)
    si_d = torch.randint(I, size=(rows, S)).to(dev)
    model.eval()

    rank_graph = {}

    def rank_and_sum(pred, flushed=False):
        """all metrics @5 of every user + their sums over users: ONE ranker launch (dccf_rank_eval_multi).  Timed as a
        CUDA-graph replay of that launch: the kernel takes ~10 us, less than the Python path to it (tensor allocation,
        ctypes marshalling), which CUDA events would otherwise count while the GPU sits idle after the flush."""
        if not flushed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            sums = rank_sums_device(pred, Y_d, iid_d, cand_d, off_d, [5])[0]
            e1.record()
            return sums, (e0, e1)
        if not rank_graph:
            rank_graph['pred'] = torch.empty_like(pred)
            rank_sums_device(rank_graph['pred'], Y_d, iid_d, cand_d, off_d, [5])        # warm (workspace, module)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode='thread_local'):
                rank_graph['sums'] = rank_sums_device(rank_graph['pred'], Y_d, iid_d, cand_d, off_d, [5])
            rank_graph['g'] = g
        rank_graph['pred'].copy_(pred)
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rank_graph['g'].replay()
        e1.record()
        return rank_graph['sums'][0], (e0, e1)

    def run_resident():
        """ids and confounder draws already in HBM; one CUDA-event pair per batch, L2 flushed in between"""
        preds, ev_pairs = [], []
        for a, b in bounds:
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            preds.append(model.predict({'X': X_d[a:b], 'rank': 1, 'train': False, 'dropout': 0.0,
                                        'sample_item': si_d[a:b]})['prediction'])
            e1.record()
            ev_pairs.append((e0, e1))
        pred = torch.cat(preds)
        sums, ev = rank_and_sum(pred, flushed=True)
        return sums, ev_pairs + [ev], pred

    def run_from_host(X_pin):
        """public API: ids from pinned host memory, confounders drawn on the torch CPU generator per batch
        (src/models/DCCF.py:72) by predict_many's worker thread, metric sums read back"""
        fds = [{'X': X_pin[a:b].to(dev, non_blocking=True), 'rank': 1, 'train': False, 'dropout': 0.0}
               for a, b in bounds]
        preds = model.predict_many(fds)
        sums, _ = rank_and_sum(torch.cat(preds))
        return sums.cpu().numpy()

    # warm-up (also loads the ranker's module: CUDA loads kernels lazily on first launch)
    for _ in range(3):
        model.predict({'X': X_d[:EVAL_BATCH], 'rank': 1, 'train': False, 'dropout': 0.0,
                            'sample_item': si_d[:EVAL_BATCH]})
        rank_sums_device(torch.zeros(rows, device=dev), Y_d, iid_d, cand_d, off_d, [5])
    # two timed passes, the faster one reported: a pass is 63 short timed regions, and a single host-side hiccup between
    # two of them (seen: ~100 ms once in several runs, in either the resident or the end-to-end pass) would otherwise be
    # charged to the kernels
    best = None
    for _ in range(2):
        barrier(world)
        sums, evs, pred = run_resident()
        barrier(world)
        s_ms = sum(a.elapsed_time(b) for a, b in evs[:-1])
        r_ms = evs[-1][0].elapsed_time(evs[-1][1])
        if best is None or s_ms + r_ms < best[0] + best[1]:
            best = (s_ms, r_ms)
    score_ms, rank_ms = best
    outputs = None
    if keep_outputs:            # the last resident pass: every candidate's score, metric sums @5 over this rank's users
        outputs = {'eval_prediction': pred.cpu().numpy(), 'eval_metrics': (sums / n_users).cpu().numpy()}
    dev_ms = dist_max(score_ms + rank_ms, world)

    # e2e: ids from pinned host memory, confounders drawn on the CPU generator per batch (as the reference),
    # metric sums read back at the end
    X_pin = torch.from_numpy(X).pin_memory()
    barrier(world)
    run_from_host(X_pin)                       # warm the pinned-buffer cache
    e2e_s = None
    for _ in range(2):
        barrier(world)
        t0 = time.perf_counter()
        host_sums = run_from_host(X_pin)
        t1 = time.perf_counter()
        e2e_s = (t1 - t0) if e2e_s is None else min(e2e_s, t1 - t0)
    e2e_s = dist_max(e2e_s, world)
    flush_s = 0.0
    metrics = host_sums / n_users
    return {'dev_ms': dev_ms, 'score_ms': score_ms, 'rank_ms': rank_ms, 'e2e_s': e2e_s, 'rows': rows,
            'n_batches': len(bounds), 'h2d': rows * 16 + rows * S * 8, 'd2h': 40,
            'ndcg@5': float(metrics[0]), 'recall@5': float(metrics[3]), 'precision@5': float(metrics[2]),
            'flush_s': flush_s, 'outputs': outputs}


# ------------------------------------------------------------------------------------------------
# noise-free evaluation (--std 0): the gather scorer, the HBM / L2-bound regime of SURVEY.md §8d
# ------------------------------------------------------------------------------------------------
# algorithmic bytes per pair when the noise-free terms come from the projected tables: ids + confounder ids, user
# row, PF row, Z PI rows, Z exposure values
BYTES_PAIR_GATHER = 16 + 8 * S + 4 * D + 4 * D + 4 * D * Z + 4 * Z


def graph_pass_ms(run_pass, replays=5):
    """Device time of one evaluation pass (all batches + ranking) replayed as ONE CUDA graph: with kernels of 10-50 us
    the eager loop measures the Python launch path, not the device.  No L2 flush inside the graph — a pass reads more
    distinct bytes than the 126 MB L2 holds (98 MB of ids + 360 MB of exposure sectors per 1 024 users at the
    electronics shape), the 8 MB of projected tables are meant to stay resident.  Returns None if capture fails."""
    try:
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, capture_error_mode='thread_local'):
            run_pass()
        for _ in range(2):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(replays):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / replays
    except Exception:       # noqa: BLE001 — the eager timing stands on its own
        return None


def noise_free_eval(U, I, n_users, dev):
    """Same evaluation workload (n_users x 1001 candidates, batches of 16384 pairs, on-device ranking) for a model
    with --std 0: scoring is dccf_score_gather.  Returns the object reported as `eval_noise_free`.  Runs in its own
    process (see main): the kernel had not run on hardware when the round's GPU budget ended."""
    from dccf_b200.models.BaseModel import candidate_layout, rank_sums_device
    model = build_model(U, I, dev, std=0.0)
    model.eval()
    flush = L2Flusher(dev)
    X, uid, iid, Y = synth_eval_set(n_users, U, I, SEED)
    rows = X.shape[0]
    bounds = [(a, min(rows, a + EVAL_BATCH)) for a in range(0, rows, EVAL_BATCH)]
    cand, off = candidate_layout(uid)
    cand_d, off_d = (None if cand is None else torch.from_numpy(cand).to(dev)), torch.from_numpy(off).to(dev)
    Y_d, iid_d, X_d = torch.from_numpy(Y).to(dev), torch.from_numpy(iid).to(dev), torch.from_numpy(X).to(dev)
    torch.manual_seed(SEED + 13)
    si_d = torch.randint(I, size=(rows, S)).to(dev)

    def fd(a, b):
        return {'X': X_d[a:b], 'rank': 1, 'train': False, 'dropout': 0.0, 'sample_item': si_d[a:b]}

    # parity of the first batch against the general FP32 scorer (the path validated against the reference)
    model.use_gather_scorer = False
    want = model.predict(fd(*bounds[0]))['prediction']
    model.use_gather_scorer = True
    got = model.predict(fd(*bounds[0]))['prediction']
    torch.cuda.synchronize()
    model.check_ids()
    rel = float((got - want).abs().max() / want.abs().max())

    def run():
        preds, evs = [], []
        for a, b in bounds:
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            preds.append(model.predict(fd(a, b))['prediction'])
            e1.record()
            evs.append((e0, e1))
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        sums = rank_sums_device(torch.cat(preds), Y_d, iid_d, cand_d, off_d, [5])[0]
        r1.record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs), r0.elapsed_time(r1), sums.cpu().numpy()

    for _ in range(3):
        run()
    eager_score_ms, rank_ms, sums = run()

    def score_only():
        return [model.predict(fd(a, b))['prediction'] for a, b in bounds]

    def whole_pass():
        return rank_sums_device(torch.cat(score_only()), Y_d, iid_d, cand_d, off_d, [5])[0]

    graph_score_ms = graph_pass_ms(score_only)
    graph_total_ms = graph_pass_ms(whole_pass)
    score_ms = graph_score_ms if graph_score_ms is not None else eager_score_ms
    total_ms = graph_total_ms if graph_total_ms is not None else eager_score_ms + rank_ms
    hbm_peak, _, peak_src = measured_peaks()
    # L2 read rate of this GPU, measured here: sum over an L2-resident 32 MiB tensor, best of 20 (a torch reduction: a
    # floor of the L2 roof, not the roof itself)
    probe = torch.ones(8 * 1024 * 1024, dtype=torch.float32, device=dev)
    best = 1e9
    for _ in range(20):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        probe.sum()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    l2_gbs = probe.numel() * 4 / 1e9 / (best / 1e3)
    pairs_per_batch = min(rows, EVAL_BATCH)
    flushed_ms = eager_score_ms / len(bounds)           # CUDA events per batch, L2 flushed before every batch
    warm_ms = score_ms / len(bounds)                    # batches back to back inside one graph (tables L2-resident)
    alg_gb = pairs_per_batch * BYTES_PAIR_GATHER / 1e9
    traffic = NCU_R2['k_gather_scores'] if pairs_per_batch == 16384 else None
    roof = {'kernel': 'k_gather_scores', 'bound': 'hbm', 'achieved': alg_gb / (flushed_ms / 1e3), 'peak': hbm_peak,
            'unit': 'GB/s', 'frac': alg_gb / (flushed_ms / 1e3) / hbm_peak, 'traffic': traffic,
            'traffic_source': NCU_R2['source'], 'peak_source': peak_src, 'bytes_per_pair': BYTES_PAIR_GATHER,
            'note': 'achieved = algorithmic bytes per batch (ids 96, user row 256, PF row 256, 11 PI rows 2816, 11 exposure '
                    'values 44 = 3468 B per pair) / time per batch with the L2 FLUSHED before every batch.  Most of those '
                    'bytes are gathers from the two projected tables (2 x I x 256 B = 8 MB), which L2 serves: DRAM sees '
                    '`traffic` (ids, exposure sectors, first touch of the tables) — the `dram` object; the `l2` object '
                    'rates the algorithmic bytes against an L2 read rate measured in this process',
            'dram': {'achieved': (traffic / 1e9 / (flushed_ms / 1e3)) if traffic else None, 'peak': hbm_peak, 'unit': 'GB/s',
                     'frac': (traffic / 1e9 / (flushed_ms / 1e3) / hbm_peak) if traffic else None},
            'l2': {'achieved': alg_gb / (flushed_ms / 1e3), 'peak': l2_gbs, 'unit': 'GB/s',
                   'frac': alg_gb / (flushed_ms / 1e3) / l2_gbs,
                   'peak_source': 'torch.sum over an L2-resident 32 MiB tensor, best of 20, this process'},
            'warm': {'ms_per_batch': warm_ms, 'achieved': alg_gb / (warm_ms / 1e3), 'unit': 'GB/s',
                     'frac_of_hbm': alg_gb / (warm_ms / 1e3) / hbm_peak, 'frac_of_l2': alg_gb / (warm_ms / 1e3) / l2_gbs,
                     'note': 'all batches of the pass replayed as one CUDA graph, no flush in between'}}
    return {'metric': 'eval_users_per_s', 'value': n_users / (total_ms / 1e3), 'unit': 'users/s',
            'config': 'same evaluation workload with --std 0 (no feature noise): dccf_score_gather + dccf_rank_eval_multi '
                      '(DCCF.use_gather_scorer, the default for noise-free inference)',
            'timing': ('one CUDA graph per pass (scoring of all batches + ranking), inputs larger than L2'
                       if graph_total_ms is not None else 'eager loop, CUDA events per batch, L2 flushed between batches'),
            'users': n_users, 'candidates_per_user': 1 + TEST_NEG_N, 'ms_per_batch': warm_ms,
            'flushed_ms_per_batch': flushed_ms, 'value_flushed': n_users / ((eager_score_ms + rank_ms) / 1e3),
            'pass_ms': total_ms, 'rank_ms': rank_ms, 'max_rel_diff_vs_general_scorer': rel, 'parity_ok': bool(rel < 1e-5),
            'roofline': roof,
            'ndcg@5': float(sums[0] / n_users), 'recall@5': float(sums[3] / n_users),
            'precision@5': float(sums[2] / n_users)}


def projected_noise_eval(U, I, n_users, dev):
    """Same evaluation workload, reference defaults (std 0.1), with DCCF.eval_noise = 'projected': the feature noise is
    drawn in the 64-dimensional image of W_f (identically distributed predictions, 64 instead of 768 normals per
    predictor row) and goes through the same tcgen05 scorer with a 64-wide operand.  Reported NEXT TO the headline
    `eval` object, which keeps the reference's formulation."""
    from dccf_b200.models.BaseModel import candidate_layout, rank_sums_device
    model = build_model(U, I, dev)
    model.eval()
    flush = L2Flusher(dev)
    X, uid, iid, Y = synth_eval_set(n_users, U, I, SEED)
    rows = X.shape[0]
    bounds = [(a, min(rows, a + EVAL_BATCH)) for a in range(0, rows, EVAL_BATCH)]
    cand, off = candidate_layout(uid)
    cand_d, off_d = (None if cand is None else torch.from_numpy(cand).to(dev)), torch.from_numpy(off).to(dev)
    Y_d, iid_d, X_d = torch.from_numpy(Y).to(dev), torch.from_numpy(iid).to(dev), torch.from_numpy(X).to(dev)
    torch.manual_seed(SEED + 13)
    si_d = torch.randint(I, size=(rows, S)).to(dev)

    def run(mode):
        model.eval_noise = mode
        preds, evs = [], []
        for a, b in bounds:
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            preds.append(model.predict({'X': X_d[a:b], 'rank': 1, 'train': False, 'dropout': 0.0,
                                        'sample_item': si_d[a:b]})['prediction'])
            e1.record()
            evs.append((e0, e1))
        pred = torch.cat(preds)
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        sums = rank_sums_device(pred, Y_d, iid_d, cand_d, off_d, [5])[0]
        r1.record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs), r0.elapsed_time(r1), sums.cpu().numpy(), pred

    for _ in range(3):
        run('projected')
    eager_score_ms, rank_ms, sums, pred_p = run('projected')
    _, _, _, pred_e = run('exact')
    model.check_ids()
    model.eval_noise = 'projected'

    def score_only():
        return [model.predict({'X': X_d[a:b], 'rank': 1, 'train': False, 'dropout': 0.0,
                               'sample_item': si_d[a:b]})['prediction'] for a, b in bounds]

    def whole_pass():
        return rank_sums_device(torch.cat(score_only()), Y_d, iid_d, cand_d, off_d, [5])[0]

    graph_score_ms = graph_pass_ms(score_only)
    graph_total_ms = graph_pass_ms(whole_pass)
    score_ms = graph_score_ms if graph_score_ms is not None else eager_score_ms
    total_ms = graph_total_ms if graph_total_ms is not None else eager_score_ms + rank_ms
    # the two modes draw different noise: predictions differ row by row but have the same distribution.  Reported:
    # mean and standard deviation over all scored rows, and the spread of the row-wise difference
    stats = {'mean_exact': float(pred_e.mean()), 'mean_projected': float(pred_p.mean()),
             'std_exact': float(pred_e.std()), 'std_projected': float(pred_p.std()),
             'rowwise_diff_std': float((pred_e - pred_p).std())}
    # end to end through the public API (predict_many from pinned host ids, metric sums read back): with the host
    # draw of the confounders (torch CPU generator replayed by dccf_confounder_draw, shipped per batch) and with the
    # generator continued on the device (DCCF.device_confounders)
    X_pin = torch.from_numpy(X).pin_memory()

    def from_host():
        fds = [{'X': X_pin[a:b].to(dev, non_blocking=True), 'rank': 1, 'train': False, 'dropout': 0.0} for a, b in bounds]
        pred = torch.cat(model.predict_many(fds))
        return rank_sums_device(pred, Y_d, iid_d, cand_d, off_d, [5])[0].cpu().numpy()

    e2e = {}
    for name, flag in (('host_draw', False), ('device_draw', True)):
        try:
            model.device_confounders = flag
            from_host()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            from_host()
            e2e[name] = {'value': n_users / (time.perf_counter() - t0), 'unit': 'users/s'}
        except Exception as exc:        # noqa: BLE001
            e2e[name] = {'error': '%s: %s' % (type(exc).__name__, str(exc)[:200])}
    model.device_confounders = False
    _, bf16_peak, peak_src = measured_peaks()
    tf32_peak = bf16_peak / 2.0
    tflop = 3 * rows * R * 2.0 * D * D / 1e12
    return {'metric': 'eval_users_per_s', 'value': n_users / (total_ms / 1e3), 'unit': 'users/s',
            'config': 'same evaluation workload, std 0.1, feature noise drawn in the 64-d image of W_f '
                      '(DCCF.eval_noise = projected): identically distributed predictions, opt-in',
            'timing': ('one CUDA graph per pass (scoring of all batches + ranking), inputs larger than L2'
                       if graph_total_ms is not None else 'eager loop, CUDA events per batch, L2 flushed between batches'),
            'users': n_users, 'candidates_per_user': 1 + TEST_NEG_N, 'ms_per_batch': score_ms / len(bounds),
            'eager_ms_per_batch': eager_score_ms / len(bounds), 'pass_ms': total_ms,
            'rank_ms': rank_ms, 'prediction_stats': stats, 'e2e': e2e,
            'roofline': {'kernel': 'k_row_scores_tc (64-wide operand)', 'bound': 'tensor',
                         'achieved': tflop / 3 / (score_ms / 1e3), 'peak': tf32_peak, 'unit': 'TFLOP/s',
                         'frac': tflop / 3 / (score_ms / 1e3) / tf32_peak,
                         'achieved_issued': tflop / (score_ms / 1e3), 'frac_issued': tflop / (score_ms / 1e3) / tf32_peak,
                         'traffic': NCU_R2['k_row_scores_tc_64'] if min(rows, EVAL_BATCH) == 16384 else None,
                         'traffic_source': NCU_R2['source'],
                         'peak_source': peak_src + ': bf16 burst / 2 for kind::tf32',
                         'hbm': {'achieved': rows * BYTES_PAIR_GATHER / 1e9 / (score_ms / 1e3), 'unit': 'GB/s',
                                 'bytes_per_pair': BYTES_PAIR_GATHER}},
            'ndcg@5': float(sums[0] / n_users), 'recall@5': float(sums[3] / n_users),
            'precision@5': float(sums[2] / n_users)}


EXTRA_LEGS = {'eval_noise_free': noise_free_eval, 'eval_projected_noise': projected_noise_eval}


def extra_legs_subprocess(preset, n_users, legs, timeout_s=420):
    """Run the legs that had not run on hardware when round 1's GPU budget ended in a CHILD process and return
    {leg: object or {'error': ...}}: a fault there must not cost the bench line of the paths that have."""
    cmd = [sys.executable, os.path.abspath(__file__), '--extra-legs-only', '--preset', preset, '--eval-users',
           str(n_users), '--legs', legs]
    legs_wanted = set(legs.split(','))
    out, err, rc = '', '', None
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, cwd=ROOT)
        out, err, rc = r.stdout, r.stderr, r.returncode
    except subprocess.TimeoutExpired as e:
        out = e.stdout.decode() if isinstance(e.stdout, bytes) else (e.stdout or '')
        err = 'timed out after %d s' % timeout_s
    legs = {}
    for ln in out.splitlines():
        if ln.startswith('{"leg"'):
            try:
                o = json.loads(ln)
                legs[o.pop('leg')] = o
            except ValueError:
                pass
    for name in EXTRA_LEGS:
        if {'eval_noise_free': 'noise_free', 'eval_projected_noise': 'projected'}[name] in legs_wanted:
            legs.setdefault(name, {'error': 'rc=%s: %s' % (rc, err[-300:])})
    return legs


# ------------------------------------------------------------------------------------------------
# CPU arm: eager-PyTorch port of the reference path on the host cores (oracle/torch_port.py)
# ------------------------------------------------------------------------------------------------
def host_threads():
    """All host cores for the CPU arm, also under torchrun (which exports OMP_NUM_THREADS=1 to every rank)."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0)) or n
    except (AttributeError, OSError):
        pass
    torch.set_num_threads(n)
    return n


def cpu_arm(U, I, X_all, budget_s, steps=None, warmup=1, eval_rows=4096):
    from oracle import torch_port
    host_cores = host_threads()
    threads = torch.get_num_threads()
    g = torch.Generator(device='cpu').manual_seed(SEED + 5)
    feat = torch.randn((I, F), generator=g) / (F ** 0.5)
    expo = torch.rand((U, I), generator=torch.Generator(device='cpu').manual_seed(SEED + 6))
    model = torch_port.DCCFPort(U, I, feat, expo, sample_num=S, attribute_num=A, std=STD, seed=SEED)
    optim = torch.optim.Adam(model.parameters(), lr=LR, weight_decay=L2)
    Y = torch.cat([torch.ones(BATCH), torch.zeros(BATCH)])
    model.train()
    times = []
    i = 0
    t_begin = time.perf_counter()
    while True:
        fd = {'X': torch.from_numpy(X_all[i % len(X_all)]), 'Y': Y, 'dropout': DROPOUT}
        t0 = time.perf_counter()
        torch_port.fit_step(model, optim, fd, L2)
        t1 = time.perf_counter()
        if i >= warmup:
            times.append(t1 - t0)
        i += 1
        if steps is not None:
            if len(times) >= steps:
                break
        elif time.perf_counter() - t_begin > budget_s and len(times) >= 2:
            break
    train_sps = BATCH * len(times) / sum(times)
    # evaluation sample: eval_rows candidate rows (≈ eval_rows/1001 users), scoring + host ranking
    Xe, uid, iid, Yl = synth_eval_set(max(1, eval_rows // (1 + TEST_NEG_N)), U, I, SEED)
    model.eval()
    with torch.no_grad():
        t0 = time.perf_counter()
        pred = model.predict({'X': torch.from_numpy(Xe), 'dropout': 0.0})['prediction'].numpy()
        torch_port.evaluate_users(pred, uid, iid, Yl, 5)
        t1 = time.perf_counter()
    n_eval_users = len(set(uid.tolist()))
    return {'train_samples_per_s': train_sps, 'train_steps': len(times), 'warmup': warmup,
            'eval_users_per_s': n_eval_users / (t1 - t0), 'eval_users': n_eval_users, 'cores': threads,
            'host_cores': host_cores}


CPU_ARM_NOTE = ('device math of the reference path only (src/models/DCCF.py:66-127 + BaseRunner.fit:175-188 as the same ATen '
                'calls, oracle/torch_port.py, validated against reference fixtures): the reference is Python with hard-coded '
                'CUDA and cannot travel to this box.  NOT included: the reference\'s host pipeline — the per-interaction Python '
                'negative sampler (src/data_processor/DataProcessor.py:446-524) and the pandas ranking of '
                'src/models/BaseModel.py:83-112 — which SURVEY.md §6 measured as the larger part of its wall time; the '
                'reference end to end is therefore slower than this number')


# ------------------------------------------------------------------------------------------------
# roofline objects
# ------------------------------------------------------------------------------------------------
def train_roofline(tr, U, I, hbm_peak, tf32_peak, peak_src):
    """Roofline of the dominant kernel of the captured step + per-kernel table.  `achieved` / `frac` count ALGORITHMIC
    work (SURVEY.md §8d: forward 2.349 MFLOP, backward 2.526 MFLOP per pair; 24 B per parameter for the sweep);
    `achieved_issued` / `frac_issued` the three TF32 products the tensor cores execute per FP32 product."""
    pairs = 2 * BATCH
    n_rows = pairs * R
    n_params = (U + I) * D + D * (D + F) + D
    if tr['kernels_us']:
        ku = tr['kernels_us']
        n_touched = pairs * (1 + Z)                      # upper bound of the rows the step touches
        work = {
            'k_train_fwd_tc': {'tensor_gflop': 3 * 2.0 * n_rows * (D + F) * D / 1e9, 'gflop': pairs * FLOP_FWD_PAIR / 1e9,
                               'mbytes': pairs * BYTES_PAIR / 1e6},
            'k_train_bwd_tc': {'tensor_gflop': 3 * 2.0 * n_rows * (D + F + 1) * D / 1e9, 'gflop': pairs * FLOP_BWD_PAIR / 1e9,
                               'mbytes': (pairs * BYTES_PAIR + 4.0 * n_rows * D) / 1e6},
            'k_adam_untouched': {'mbytes': 24.0 * ((U + I) * D - n_touched * D) / 1e6},
            'k_adam_touched': {'mbytes': 24.0 * (n_touched * D + D * (D + F) + D) / 1e6},
            'k_train_mid': {'mbytes': (4.0 * 3 * n_rows * D + 4.0 * n_rows * D) / 1e6},
        }
        kernels_obj = {}
        for name, k in ku.items():
            o = {'us': k['us'], 'start_us': k['start_us'], 'end_us': k['end_us']}
            w = work.get(name, {})
            if 'mbytes' in w:
                o['mbytes'] = w['mbytes']
                o['gbs'] = w['mbytes'] / 1e3 / (k['us'] / 1e6) if k['us'] > 0 else 0.0
            if 'gflop' in w:
                o['gflop'] = w['gflop']
                o['algorithmic_tflops'] = w['gflop'] / 1e3 / (k['us'] / 1e6)
                o['issued_tf32_tflops'] = w['tensor_gflop'] / 1e3 / (k['us'] / 1e6)
            kernels_obj[name] = o
        for name, tb in NCU_TRAFFIC_BYTES.items():
            if name in kernels_obj:
                kernels_obj[name]['dram_traffic_mbytes'] = tb / 1e6
        crit = [n_ for n_ in ('k_train_fwd_tc', 'k_train_mid', 'k_train_bwd_tc', 'k_adam_touched') if n_ in ku]
        dom = max(crit, key=lambda n_: ku[n_]['us'])
        d = kernels_obj[dom]
        if 'algorithmic_tflops' in d:
            roof = {'kernel': dom + ' (tcgen05 3xTF32)', 'bound': 'tensor', 'achieved': d['algorithmic_tflops'],
                    'peak': tf32_peak, 'unit': 'TFLOP/s', 'frac': d['algorithmic_tflops'] / tf32_peak,
                    'achieved_issued': d['issued_tf32_tflops'], 'frac_issued': d['issued_tf32_tflops'] / tf32_peak,
                    'traffic': NCU_TRAFFIC_BYTES.get(dom), 'traffic_source': NCU_TRAFFIC_SOURCE,
                    'peak_source': peak_src + ': bf16 burst / 2 for kind::tf32',
                    'work_note': 'achieved / frac = algorithmic flops of the reference formulation (SURVEY.md §8d) per launch / '
                                 'kernel time; *_issued = the 3 TF32 products per FP32 product actually executed',
                    'limiter': 'the operand tile is generated, not loaded (Philox4x32-10 + Box-Muller, 4.3 M normals per step in '
                               'each of the two contractions, 16 producer warps per SM): latency of the producer loop, not the '
                               'tensor pipe or HBM',
                    'fp32_simt': {'achieved': d['algorithmic_tflops'], 'peak': FP32_PEAK_TFLOPS, 'unit': 'TFLOP/s',
                                  'frac': d['algorithmic_tflops'] / FP32_PEAK_TFLOPS}}
        else:
            roof = {'kernel': dom, 'bound': 'hbm', 'achieved': d.get('gbs', 0.0), 'peak': hbm_peak, 'unit': 'GB/s',
                    'frac': d.get('gbs', 0.0) / hbm_peak, 'traffic': NCU_TRAFFIC_BYTES.get(dom),
                    'traffic_source': NCU_TRAFFIC_SOURCE, 'peak_source': peak_src}
        sweep = kernels_obj.get('k_adam_untouched')
        if sweep is not None:
            roof['side_stream_sweep'] = {'kernel': 'k_adam_untouched', 'bound': 'hbm', 'achieved': sweep['gbs'],
                                         'peak': hbm_peak, 'unit': 'GB/s', 'frac': sweep['gbs'] / hbm_peak,
                                         'note': 'l2 + clip + Adam over the untouched rows on a side stream, one small CTA per SM '
                                                 'beside the tensor-core kernels (128 threads; 256 under data parallelism); '
                                                 'off the critical path by design, so its rate is a floor, not a target'}
        step_us = tr['timeline_step_us']
        roof['whole_step'] = {'us': step_us, 'hbm_frac': 24.0 * n_params / 1e9 / (step_us / 1e6) / hbm_peak if step_us else None,
                              'fp32_simt_frac': pairs * (FLOP_FWD_PAIR + FLOP_BWD_PAIR) / 1e12 / (step_us / 1e6) / FP32_PEAK_TFLOPS
                              if step_us else None,
                              'note': 'algorithmic bytes (24 B per parameter) and flops (forward + backward) of the whole step '
                                      'over the step length by the same stamps'}
        roof['kernels_note'] = ('per-kernel %%globaltimer stamps inside extra replays of the captured step, L2 flushed '
                                'before each measured step; step length by the same stamps: %.1f us' % step_us)
        roof['kernels'] = kernels_obj
        return roof
    stage = tr['stage_ms']                               # fwd, bwd, adam  (ms per step)
    stages = {
        'score_fwd': {'ms': float(stage[0]), 'gflop': pairs * FLOP_FWD_PAIR / 1e9, 'mbytes': pairs * BYTES_PAIR / 1e6},
        'bpr_bwd': {'ms': float(stage[1]), 'gflop': pairs * FLOP_BWD_PAIR / 1e9,
                    'mbytes': pairs * (BYTES_PAIR + 4 * D * (1 + Z)) / 1e6},
        'adam_sweep': {'ms': float(stage[2]), 'gflop': 0.0, 'mbytes': 24.0 * n_params / 1e6},
    }
    for st in stages.values():
        st['gbs'] = st['mbytes'] / 1e3 / (st['ms'] / 1e3) if st['ms'] > 0 else 0.0
        st['tflops'] = st['gflop'] / 1e3 / (st['ms'] / 1e3) if st['ms'] > 0 else 0.0
    dom = max(stages, key=lambda k: stages[k]['ms'])
    return {'kernel': dom, 'bound': 'hbm', 'achieved': stages[dom]['gbs'], 'peak': hbm_peak, 'unit': 'GB/s',
            'frac': stages[dom]['gbs'] / hbm_peak, 'traffic': None, 'peak_source': peak_src,
            'fp32_simt': {'achieved': stages[dom]['tflops'], 'peak': FP32_PEAK_TFLOPS, 'unit': 'TFLOP/s',
                          'frac': stages[dom]['tflops'] / FP32_PEAK_TFLOPS},
            'stages_note': 'per-stage CUDA events of the same step launched kernel by kernel (includes launch gaps; '
                           'the timed value replays the step as one CUDA graph)',
            'stages': stages}


def eval_object(model, evl, n_users_total, world, hbm_peak, tf32_peak, peak_src):
    eval_pairs = evl['rows']
    eval_users_s = n_users_total / (evl['dev_ms'] / 1e3)
    eval_tflops = eval_pairs * FLOP_FWD_PAIR / 1e12 / (evl['score_ms'] / 1e3)
    used_tc = bool(getattr(model, 'use_tensor_cores', False)) and eval_pairs * R >= model.tc_min_rows
    noise_tflop = 3 * eval_pairs * R * 2.0 * F * D / 1e12          # the three TF32 products actually issued
    hbm = {'achieved': eval_pairs * BYTES_PAIR / 1e9 / (evl['score_ms'] / 1e3), 'peak': hbm_peak, 'unit': 'GB/s',
           'frac': eval_pairs * BYTES_PAIR / 1e9 / (evl['score_ms'] / 1e3) / hbm_peak}
    if used_tc:
        eval_roof = {'kernel': 'k_row_scores_tc (tcgen05 3xTF32)', 'bound': 'tensor',
                     'achieved': eval_tflops, 'peak': tf32_peak, 'unit': 'TFLOP/s', 'frac': eval_tflops / tf32_peak,
                     'achieved_issued': noise_tflop / (evl['score_ms'] / 1e3),
                     'frac_issued': noise_tflop / (evl['score_ms'] / 1e3) / tf32_peak,
                     'traffic': NCU_EVAL_TRAFFIC_BYTES if EVAL_BATCH == 16384 else None,
                     'traffic_source': NCU_EVAL_TRAFFIC_SOURCE,
                     'peak_source': peak_src + ': bf16 burst / 2 for kind::tf32',
                     'work_note': 'achieved / frac = algorithmic FP32 flops of the reference formulation (2.349 MFLOP per pair) / '
                                  'scoring time; *_issued = the 3 TF32 products per FP32 product actually executed',
                     'limiter': 'Gaussian noise generation (Philox4x32-10 + Box-Muller, 16.9 M normals per user) on '
                                'the SIMT ALU/XU pipes, not the tensor pipe',
                     'fp32_simt': {'achieved': eval_tflops, 'peak': FP32_PEAK_TFLOPS, 'unit': 'TFLOP/s',
                                   'frac': eval_tflops / FP32_PEAK_TFLOPS,
                                   'note': 'the same algorithmic flops against the FP32 SIMT peak a non-tensor-core kernel is '
                                           'bounded by'},
                     'hbm': hbm}
    else:
        eval_roof = dict(hbm, kernel='k_row_scores', bound='hbm', traffic=None,
                         fp32_simt={'achieved': eval_tflops, 'peak': FP32_PEAK_TFLOPS, 'unit': 'TFLOP/s',
                                    'frac': eval_tflops / FP32_PEAK_TFLOPS})
    rank_bytes = 8.0 * eval_pairs
    return {'metric': 'eval_users_per_s', 'value': eval_users_s, 'unit': 'users/s',
            'users': n_users_total, 'candidates_per_user': 1 + TEST_NEG_N,
            'timing': 'CUDA events per 16384-pair batch (L2 flushed before each) + the ranker launch; the faster of two passes, '
                      'for the device-resident number and for the end-to-end one',
            'ms_per_batch': evl['score_ms'] / evl['n_batches'], 'rank_ms': evl['rank_ms'],
            'ranker': {'kernel': 'k_rank_stream (one pass, all metrics, one launch)', 'ms': evl['rank_ms'], 'bound': 'hbm',
                       'achieved': rank_bytes / 1e9 / (evl['rank_ms'] / 1e3), 'peak': hbm_peak, 'unit': 'GB/s',
                       'frac': rank_bytes / 1e9 / (evl['rank_ms'] / 1e3) / hbm_peak,
                       'traffic': NCU_R2['k_rank_stream'] if eval_pairs == 1024 * (1 + TEST_NEG_N) else None,
                       'traffic_source': NCU_R2['source'],
                       'note': 'algorithmic bytes = 8 B per candidate (score + label) of this rank; CUDA events around the '
                               'launch, L2 flushed before it'},
            'e2e': {'value': n_users_total / evl['e2e_s'], 'unit': 'users/s',
                    'h2d_bytes': evl['h2d'], 'd2h_bytes': evl['d2h']},
            'roofline': eval_roof,
            'ndcg@5': evl['ndcg@5'], 'recall@5': evl['recall@5'], 'precision@5': evl['precision@5']}


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--preset', default='electronics', choices=sorted(PRESETS))
    ap.add_argument('--eval-users', type=int, default=1024)
    ap.add_argument('--cpu-budget', type=float, default=12.0, help='seconds of CPU work for the cpu_baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extra-legs', action='store_true',
                    help='skip every leg beyond the headline train / eval pair (and the data-parallel parity check)')
    ap.add_argument('--legs', default='all',
                    help='comma list of: config3,config4,config5,eager,noise_free,projected (default all that apply)')
    ap.add_argument('--extra-legs-only', action='store_true', help='run only the child-process legs, one JSON line each')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed training step (prediction, loss, the '
                         'parameters it left) and the last timed evaluation pass (predictions, metrics @5) computed, '
                         'as DIR/<name>.npy (rank 0; inputs are seeded, so two builds can be compared array by array)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes what the GPU path computed: not available with --impl reference')
    args.warmup = max(args.warmup, 3)
    U, I = PRESETS[args.preset]
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    legs = set(['config3', 'config4', 'config5', 'eager', 'noise_free', 'projected']) if args.legs == 'all' else \
        set(x for x in args.legs.split(',') if x)
    if args.no_extra_legs:
        legs = set()

    def workload(preset, U_, I_):
        return {'workload': 'DCCF Adam lr=1e-3 on synthetic %s-shape data: U=%d I=%d F=768 D=64, batch 128 (+128 sampled '
                            'negatives) per rank, S=10 A=2 std=0.1 dropout=0.2 l2=1e-4; eval test_neg_n=1000, eval_batch 16384, '
                            'ndcg/recall/precision@5' % (preset, U_, I_),
                'preset': preset, 'users': U_, 'items': I_, 'batch_size': BATCH, 'eval_users_per_rank': args.eval_users,
                'parallelism': 'dp%d' % world, 'l2_cache': 'flushed between timed iterations (256 MiB write)'}

    config = workload(args.preset, U, I)

    if args.impl == 'reference':
        if rank != 0:
            return
        X_all = synth_batches(64, U, I, SEED)
        r = cpu_arm(U, I, X_all, budget_s=0.0, steps=args.steps, warmup=args.warmup)
        sample = '%d train steps of 128 samples after %d warm-up steps; eval of %d users x 1001 candidates' \
                 % (r['train_steps'], r['warmup'], r['eval_users'])
        line = {'impl': 'reference', 'metric': 'train_samples_per_s', 'value': r['train_samples_per_s'],
                'unit': 'samples/s', 'n_gpus': args.gpus, 'steps': r['train_steps'], 'warmup': r['warmup'],
                'ms_per_step': 1e3 * BATCH / r['train_samples_per_s'], 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': dict(config, parallelism='cpu'),
                'cpu_baseline': {'value': r['train_samples_per_s'], 'unit': 'samples/s', 'cores': r['cores'],
                                 'host_cores': r['host_cores'], 'kind': 'port', 'sample': sample, 'note': CPU_ARM_NOTE},
                'e2e': {'value': r['train_samples_per_s'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0,
                        'd2h_bytes_per_step': 0},
                'eval': {'metric': 'eval_users_per_s', 'value': r['eval_users_per_s'], 'unit': 'users/s'},
                'note': 'reference CPU path = eager-PyTorch port of src/models/DCCF.py + BaseRunner.fit '
                        '(oracle/torch_port.py) on ONE process with all host cores whatever --gpus says (a CPU arm does not '
                        'scale with the GPU count: only the N = 1 ratio is meaningful)'}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if args.extra_legs_only:
        for name, fn in EXTRA_LEGS.items():
            if {'eval_noise_free': 'noise_free', 'eval_projected_noise': 'projected'}[name] not in legs:
                continue
            try:
                o = fn(U, I, args.eval_users, dev)
            except Exception as exc:        # noqa: BLE001 — reported; a sticky CUDA error fails the next leg too
                o = {'error': '%s: %s' % (type(exc).__name__, str(exc)[:300])}
            print(json.dumps(dict(leg=name, **o)), flush=True)
        return
    if world > 1:
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'          # keep NCCL's version banner off stdout: ONE JSON line
        torch.distributed.init_process_group('nccl', device_id=dev)
    from dccf_b200 import kernels  # noqa: F401  (fails loudly here when the library is missing)
    from tools import bench_legs
    peaks = measured_peaks()
    hbm_peak, bf16_peak, peak_src = peaks
    tf32_peak = bf16_peak / 2.0          # kind::tf32 runs at half the bf16 rate

    # ---- data parallel: equality with the single-GPU step BEFORE any timing --------------------------------------
    dp_parity = None
    if world > 1:
        dp_parity = bench_legs.dp_parity_check(world, rank, dev)
        if not dp_parity['ok']:
            if rank == 0:
                print(json.dumps({'metric': 'train_samples_per_s', 'value': None, 'n_gpus': world, 'dp_parity_ok': False,
                                  'dp_parity': dp_parity, 'error': 'data-parallel step differs from the single-GPU step'}))
            torch.distributed.destroy_process_group()
            sys.exit(3)

    def train_eval(preset, steps, warmup, eval_users, keep_outputs=False):
        """The headline pair at one shape: (model, train result, eval result, clocks)."""
        U_, I_ = PRESETS[preset]
        model = build_model(U_, I_, dev)
        if world > 1:
            model.enable_data_parallel()
        flush = L2Flusher(dev)
        X_all = synth_batches(warmup + steps, U_, I_, SEED + rank)
        with ClockSampler(local_rank) as clocks:
            tr = bench_train(model, X_all, steps, warmup, world, flush, keep_outputs)
            evl = bench_eval(model, eval_users, 3, world, rank, flush, keep_outputs)
        return model, tr, evl, clocks.summary()

    keep_outputs = bool(args.dump_outputs) and rank == 0
    model, tr, evl, clk = train_eval(args.preset, args.steps, args.warmup, args.eval_users, keep_outputs)
    if keep_outputs:
        dump_outputs(args.dump_outputs, dict(tr['outputs'], **evl['outputs']))
    ms_per_step = tr['total_ms'] / args.steps
    value = world * BATCH * args.steps / (tr['total_ms'] / 1e3)
    e2e_value = world * BATCH * args.steps / tr['e2e_s']
    line = {'metric': 'train_samples_per_s', 'value': value, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config,
            'e2e': {'value': e2e_value, 'unit': 'samples/s', 'h2d_bytes_per_step': tr['h2d'],
                    'd2h_bytes_per_step': tr['d2h'],
                    'timing': 'model.train_step per step from pinned host ids: staging + confounder draw on the torch CPU '
                              'generator + one H2D copy + one CUDA-graph launch + D2H copy of the loss, every step; the host '
                              'does not wait inside the loop (one synchronise ends the timed region); wall clock minus the '
                              'device time of the L2 flushes between the steps (CUDA events around each flush)',
                    'sync_every_step': {'value': world * BATCH / tr['e2e_sync_s_per_step'], 'unit': 'samples/s',
                                        'note': 'same call, host blocked on loss.item() after every step (latency of one '
                                                'step end to end, no overlap of host and device)'}},
            'back_to_back': {'ms_per_step': tr['b2b_ms'], 'value': world * BATCH / (tr['b2b_ms'] / 1e3), 'unit': 'samples/s',
                             'note': 'same steps without the L2 flush between them (parameters stay L2-resident), one '
                                     'CUDA-event pair around all of them'},
            'gpu_launches': int(tr['launches']), 'clocks': clk,
            'roofline': train_roofline(tr, U, I, hbm_peak, tf32_peak, peak_src),
            'eval': eval_object(model, evl, world * args.eval_users, world, hbm_peak, tf32_peak, peak_src),
            'last_loss': tr['last_loss']}
    if world > 1:
        dp_parity['replicas_identical_after_timed_steps'] = bench_legs.replica_checksum(model, world, dev)
        line['dp_parity_ok'] = bool(dp_parity['ok'] and dp_parity['replicas_identical_after_timed_steps'])
        line['dp_parity'] = dp_parity
    del model
    torch.cuda.empty_cache()

    def guarded(name, fn):
        """A leg must not cost the line: its failure is reported in its own object.  (All ranks run every leg.)"""
        try:
            line[name] = fn()
        except Exception as exc:            # noqa: BLE001
            line[name] = {'error': '%s: %s' % (type(exc).__name__, str(exc)[:300])}
        torch.cuda.empty_cache()

    if 'config3' in legs and args.preset != 'cds':
        def config3():
            steps3, warm3 = min(args.steps, 100), min(args.warmup, 5)
            m3, tr3, ev3, _ = train_eval('cds', steps3, warm3, min(args.eval_users, 512))
            U3, I3 = PRESETS['cds']
            o = {'metric': 'train_samples_per_s', 'value': world * BATCH * steps3 / (tr3['total_ms'] / 1e3),
                 'unit': 'samples/s', 'n_gpus': world, 'steps': steps3, 'warmup': warm3,
                 'ms_per_step': tr3['total_ms'] / steps3, 'scaling': 'weak', 'config': workload('cds', U3, I3),
                 'e2e': {'value': world * BATCH * steps3 / tr3['e2e_s'], 'unit': 'samples/s'},
                 'back_to_back_ms_per_step': tr3['b2b_ms'],
                 'eval': {'value': world * min(args.eval_users, 512) / (ev3['dev_ms'] / 1e3), 'unit': 'users/s',
                          'ms_per_batch': ev3['score_ms'] / ev3['n_batches'], 'rank_ms': ev3['rank_ms']},
                 'last_loss': tr3['last_loss']}
            if world > 1:
                o['replicas_identical'] = bench_legs.replica_checksum(m3, world, dev)
            return o
        guarded('config3_cds', config3)
    if 'config4' in legs:
        guarded('config4_full_catalogue', lambda: bench_legs.full_catalogue_leg(world, rank, dev, peaks))
    if 'config5' in legs:
        guarded('config5_scaled', lambda: bench_legs.scaled_leg(world, rank, dev, peaks))
    if rank == 0 and world == 1:
        if 'eager' in legs:
            cfg = {'D': D, 'F': F, 'S': S, 'A': A, 'std': STD, 'seed': SEED, 'lr': LR, 'l2': L2, 'batch': BATCH,
                   'dropout': DROPOUT, 'eval_batch': EVAL_BATCH, 'test_neg_n': TEST_NEG_N}
            guarded('gpu_eager_reference', lambda: bench_legs.gpu_eager_reference(U, I, dev, cfg))
            g = line.get('gpu_eager_reference', {})
            if 'train_samples_per_s' in g:
                g['ours_over_eager'] = {'train': value / g['train_samples_per_s'],
                                        'eval_scoring': line['eval']['value'] / g['eval_users_per_s']}
        if not args.no_cpu_baseline:
            X_cpu = synth_batches(32, U, I, SEED)
            c = cpu_arm(U, I, X_cpu, budget_s=args.cpu_budget)
            line['cpu_baseline'] = {'value': c['train_samples_per_s'], 'unit': 'samples/s', 'cores': c['cores'],
                                    'host_cores': c['host_cores'], 'kind': 'port',
                                    'sample': '%d train steps of 128 samples (eager-PyTorch port of the reference path, '
                                              'oracle/torch_port.py); eval sample %d users -> %.3f users/s'
                                              % (c['train_steps'], c['eval_users'], c['eval_users_per_s']),
                                    'eval_users_per_s': c['eval_users_per_s'], 'note': CPU_ARM_NOTE}
        child = [n for n in ('noise_free', 'projected') if n in legs]
        if child:
            line.update(extra_legs_subprocess(args.preset, args.eval_users, ','.join(child)))
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
