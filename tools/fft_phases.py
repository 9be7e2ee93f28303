#!/usr/bin/env python
"""Where the CMux step of the FP64 FFT kernel (blind_rotate_fft_kernel, fft_kernels.cuh) spends its cycles, per phase.

Builds the library with -DNB_FFT_PHASE_CLOCKS into a temporary directory (never over the in-tree .so), or takes such a
build with --lib, runs gate_nand bootstraps at one batch size and reads the per-CTA clock64() sums of thread 0:
fwd1, fwd2, fwd3, MAC, inv3, inv2, inv1 (thread 0's own work in the phase), sync (its waits at the step's barriers,
i.e. the time the slowest warp took beyond thread 0's) and other (fetching the next rotation).  Reported per CTA-step,
summed over all CTAs and steps of the timed launches.  The clock reads add a few instructions and registers to the
profiling build, so its kernel time is quoted next to the phases.  Needs a GPU.

    python tools/fft_phases.py [--batch 4096] [--reps 3] [--define NB_FFT_CT=4] [--out profiles/r4_fft_phases_before.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SLOTS = ('fwd1', 'fwd2', 'fwd3', 'mac', 'inv3', 'inv2', 'inv1', 'sync', 'other', 'steps')   # FFT_CLK_* order
CTAS = 1024                                                                                    # FFT_CLK_CTAS


def build_variant(defines):
    import __graft_entry__ as g
    out = os.path.join(tempfile.mkdtemp(prefix='nb_fft_phases_'), 'libnufhe_b200.so')
    cmd = ['nvcc'] + g.NVCC_FLAGS + ['-DNB_FFT_PHASE_CLOCKS'] + ['-D' + d for d in defines] + [
        '-o', out, os.path.join(g.CSRC, 'capi.cu')]
    subprocess.check_call(cmd, cwd=g.CSRC)
    return out


def gpu_info():
    q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm',
                        '--format=csv,noheader,nounits'], capture_output=True, text=True)
    f = [x.strip() for x in q.stdout.strip().split(',')]
    return {'name': f[0], 'power_limit_w': float(f[1]), 'sm_clock_mhz': float(f[2]), 'sm_clock_max_mhz': float(f[3])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--lib', default=None, help='a library built with -DNB_FFT_PHASE_CLOCKS (default: build one)')
    ap.add_argument('--define', action='append', default=[], help='extra -D for the build, e.g. NB_FFT_CT=4')
    ap.add_argument('--batch', type=int, default=4096)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    lib_path = args.lib or build_variant(args.define)
    os.environ['NUFHE_B200_LIB'] = lib_path
    os.environ['NUFHE_B200_FFT'] = '1'
    import numpy
    import torch
    from oracle import oracle as O
    from nufhe_b200.engine import Engine
    e = Engine(0)
    read = ctypes.CDLL(lib_path).nb_fft_phase_clocks
    read.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
    buf = numpy.zeros((CTAS, len(SLOTS)), numpy.uint64)

    def take(reset):
        rc = read(e.handle, buf.ctypes.data, int(reset))
        assert rc == 0, 'nb_fft_phase_clocks failed (%d); was the library built with -DNB_FFT_PHASE_CLOCKS?' % rc
        return buf.copy()

    keys = O.OracleKeys(20261017)
    bk = e.bk_prepare(e.to_device(keys.bk))
    num, den, sa, sb = O.GATE_TABLE['nand']
    rng = numpy.random.RandomState(7)
    B = args.batch
    d = [(e.to_device(rng.randint(-2**31, 2**31, (B, 500), dtype=numpy.int32)),
          e.to_device(rng.randint(-2**31, 2**31, (B,), dtype=numpy.int32))) for _ in range(2)]
    c = O.phase_to_t32(num, den)
    e.bootstrap_extract(d[0], d[1], c, sa, sb, O.MU, bk)             # warm-up
    take(True)
    ms = []
    for _ in range(args.reps):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        e.bootstrap_extract(d[0], d[1], c, sa, sb, O.MU, bk)
        s1.record()
        torch.cuda.synchronize()
        ms.append(s0.elapsed_time(s1))
    info = gpu_info()
    clk = take(False).astype(numpy.float64)
    tot = clk.sum(axis=0)
    steps = tot[SLOTS.index('steps')]
    per_step = {s: tot[i] / steps for i, s in enumerate(SLOTS) if s != 'steps'}
    step_cycles = sum(per_step.values())
    res = {'gpu': info, 'batch': B, 'reps': args.reps, 'defines': args.define, 'lib': os.path.basename(lib_path),
           'kernel_ms': ms, 'ctas_reporting': int((clk[:, SLOTS.index('steps')] > 0).sum()),
           'cta_steps': steps, 'cycles_per_cta_step': step_cycles,
           'phases_cycles_per_cta_step': per_step,
           'phases_share': {s: v / step_cycles for s, v in per_step.items()},
           'note': 'clock64() of thread 0 of each CTA, summed over CTAs and steps; sync = waits at the step barriers'}
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
