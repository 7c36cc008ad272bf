"""Occupancy facts the training step's schedule relies on, read from the built library's resource usage (registers and
static shared memory per kernel, `cuobjdump --dump-resource-usage`) and the launch shapes below.  No GPU needed.

The dW kernel is a programmatic dependent of the middle kernel: its CTAs are placed while middle-kernel CTAs still run,
so on the few free SMs two of them could share one SM and end late.  Its resources must allow exactly one per SM, still
fit beside the side-stream sweep's CTA, and never fit beside a middle-kernel CTA (nor a forward CTA)."""
import os
import re
import shutil
import subprocess

import pytest

from dccf_b200 import build

SM_REGS = 65536
SM_SMEM = 228 * 1024            # shared memory of an SM (B200)
CTA_RESERVED_SMEM = 1024        # reserved by the system for every resident CTA
REG_ALLOC_UNIT = 256            # registers are allocated per warp in units of 256

# launch shapes: threads, dynamic shared memory
TC_RING = 2 * 48 * 1024 + 256   # TT_SMEM_BYTES (tc_train.cu)
SHAPES = {
    'k_train_fwd_tc': (576, TC_RING),        # TC_NT
    'k_train_bwd_tc': (608, TC_RING),        # TB_NT: 16 producer warps + MMA warp + 2 idle warps
    'k_train_mid': (768, 0),                 # TM_NT (its dynamic shared memory is small; not the limiter)
    'untouched': (224, 120 * 1024),          # side-stream sweep: default width, ADAM_SIDE_SMEM limiter (adam.cu)
}
SWEEPS = ('k_adam_untouched', 'k_gd_untouched', 'k_adagrad_untouched')


@pytest.fixture(scope='module')
def usage():
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    out = subprocess.run([cuobjdump, '--dump-resource-usage', build.build()], capture_output=True, text=True).stdout
    found = {}
    for name, reg, shared in re.findall(r'Function (\S+):\s*\n\s*REG:(\d+) .*?SHARED:(\d+)', out):
        found[name] = (int(reg), int(shared))
    assert found, out[:2000]

    def get(kernel):
        hits = [v for k, v in found.items() if re.search(r'\d%s' % kernel, k)]
        assert hits, kernel
        return hits

    return get


def cta(usage, kernel, shape=None):
    """Worst case over the kernel's instantiations: (registers, shared memory bytes) one resident CTA takes."""
    threads, dyn = SHAPES[shape or kernel]
    warps = (threads + 31) // 32
    regs = max(-(-reg * 32 // REG_ALLOC_UNIT) * REG_ALLOC_UNIT * warps for reg, _ in usage(kernel))
    smem = max(shared + dyn + CTA_RESERVED_SMEM for _, shared in usage(kernel))
    return regs, smem


def fits(*ctas):
    return sum(r for r, _ in ctas) <= SM_REGS and sum(s for _, s in ctas) <= SM_SMEM


def test_middle_kernel_is_capped_at_64_registers(usage):
    assert all(reg <= 64 for reg, _ in usage('k_train_mid'))


def test_one_dw_cta_per_sm(usage):
    dw = cta(usage, 'k_train_bwd_tc')
    assert not fits(dw, dw), dw


def test_dw_cta_fits_beside_every_sweep_cta(usage):
    dw = cta(usage, 'k_train_bwd_tc')
    for sweep in SWEEPS:
        assert fits(dw, cta(usage, sweep, 'untouched')), sweep


def test_dw_cta_never_shares_an_sm_with_a_middle_or_forward_cta(usage):
    dw = cta(usage, 'k_train_bwd_tc')
    assert not fits(dw, cta(usage, 'k_train_mid'))
    assert not fits(dw, cta(usage, 'k_train_fwd_tc'))


def test_middle_cta_fits_beside_every_sweep_cta_but_not_beside_a_forward_cta(usage):
    mid = cta(usage, 'k_train_mid')
    for sweep in SWEEPS:
        assert fits(mid, cta(usage, sweep, 'untouched')), sweep
    assert not fits(mid, cta(usage, 'k_train_fwd_tc'))
