#!/usr/bin/env python
"""A/B of the fused bootstrap's FP64 FFT kernel against the NTT kernel in one process: two Engines, one created with
NUFHE_B200_FFT=1 and one with 0 (the knob is read at context creation), alternated call by call on the same seeded
inputs.  Reports, per batch, the median and spread (min - max) of the fused-kernel time (CUDA events around
bootstrap_extract / bootstrap_extract2) and of gate_nand / gate_mux throughput (bootstraps + key switch), and checks
that both kernels return the same bits.  Needs a GPU.

    python tools/fft_ab.py [--batches 592 1024 4096 16384] [--reps 5] [--out profiles/r3_fft_ab.json]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batches', type=int, nargs='+', default=[592, 1024, 4096, 16384])
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import numpy
    import torch
    from oracle import oracle as O
    from nufhe_b200.engine import Engine
    engines = {}
    for knob in ('0', '1'):
        os.environ['NUFHE_B200_FFT'] = knob
        e = Engine(0)
        engines[knob] = e
    keys = O.OracleKeys(20261017)
    dk = {k: (e.bk_prepare(e.to_device(keys.bk)), (e.to_device(keys.ks_a), e.to_device(keys.ks_b), e.to_device(keys.ks_cv)))
          for k, e in engines.items()}
    num, den, sa, sb = O.GATE_TABLE['nand']
    nand_c, and_c = O.phase_to_t32(num, den), O.phase_to_t32(-1, 8)
    rng = numpy.random.RandomState(7)
    res = {'device': torch.cuda.get_device_name(0), 'batches': {}}
    for B in args.batches:
        cts = [tuple(numpy.ascontiguousarray(x) for x in (rng.randint(-2**31, 2**31, (B, 500), dtype=numpy.int32),
                                                          rng.randint(-2**31, 2**31, (B,), dtype=numpy.int32)))
               for _ in range(3)]
        row = {}
        outs = {}
        for gate in ('nand', 'mux'):
            t_k = {'0': [], '1': []}
            t_g = {'0': [], '1': []}
            for rep in range(args.reps + 1):                     # rep 0 warms up
                for knob, e in engines.items():
                    bk, ks = dk[knob]
                    d = [(e.to_device(a), e.to_device(b)) for a, b in cts]
                    torch.cuda.synchronize()
                    s0, s1, s2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                    s0.record()
                    if gate == 'nand':
                        ext = e.bootstrap_extract(d[0], d[1], nand_c, sa, sb, O.MU, bk)
                        s1.record()
                        r = e.keyswitch(ks, ext)
                    else:
                        u1, u2 = e.bootstrap_extract2((d[0], d[1], and_c, 1, 1), (d[0], d[2], and_c, -1, 1), O.MU, bk)
                        s1.record()
                        r = e.keyswitch(ks, u1, u2, c=O.phase_to_t32(1, 8))
                    s2.record()
                    torch.cuda.synchronize()
                    if rep:
                        t_k[knob].append(s0.elapsed_time(s1))
                        t_g[knob].append(s0.elapsed_time(s2))
                    outs[(gate, knob)] = (e.to_host(r[0]), e.to_host(r[1]))
            same = all((x == y).all() for x, y in zip(outs[(gate, '0')], outs[(gate, '1')]))
            for knob in ('0', '1'):
                row['%s_fft%s' % (gate, knob)] = {
                    'kernel_ms_median': statistics.median(t_k[knob]), 'kernel_ms_min': min(t_k[knob]),
                    'kernel_ms_max': max(t_k[knob]),
                    'gates_per_s_median': B / statistics.median(t_g[knob]) * 1e3,
                    'gates_per_s_min': B / max(t_g[knob]) * 1e3, 'gates_per_s_max': B / min(t_g[knob]) * 1e3}
            row['%s_same_bits' % gate] = bool(same)
            print(B, gate, 'NTT %.2f ms' % row['%s_fft0' % gate]['kernel_ms_median'],
                  'FFT %.2f ms' % row['%s_fft1' % gate]['kernel_ms_median'], 'same bits:', same, flush=True)
        res['batches'][str(B)] = row
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
