#!/bin/bash
# Round 2, final 8-GPU call: the full bench line (every leg) at 8 ranks.
mkdir -p gpurun_out
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29533"
show() {
python - "$1" <<'P'
import json, sys
try:
    d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
    k = d['roofline'].get('kernels', {})
    print(sys.argv[1], 'value', round(d['value']), 'ms/step', round(d['ms_per_step'], 5), 'b2b', round(d['back_to_back']['ms_per_step'], 5), 'e2e', round(d['e2e']['value']), 'parity', d.get('dp_parity_ok'), 'eval', round(d['eval']['value']))
    for n, o in sorted(k.items(), key=lambda kv: kv[1]['start_us']):
        print('    %-32s %6.1f -> %6.1f' % (n, o['start_us'], o['end_us']))
    for kk in ('config3_cds', 'config4_full_catalogue', 'config5_scaled'):
        if kk in d: print(kk, json.dumps(d.get(kk))[:700])
except Exception as e:
    print(sys.argv[1], 'parse failed', e)
P
}
DCCF_BENCH_RANK_TIMELINES=1 timeout 900 $TR bench.py --gpus 8 --steps 100 --warmup 5 > gpurun_out/bench_r2_dp8.json 2> gpurun_out/bench_r2_dp8.err; echo rc=$?; grep '"rank"' gpurun_out/bench_r2_dp8.err | cut -c1-700 | head -3; tail -c 300 gpurun_out/bench_r2_dp8.err; show gpurun_out/bench_r2_dp8.json
nvidia-smi --query-gpu=index,clocks.sm,clocks.max.sm,power.draw,temperature.gpu --format=csv,noheader | head -3
