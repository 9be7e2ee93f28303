#!/usr/bin/env python
"""bench.py -- headline benchmark of the nufhe_b200 engine (contract: see the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--gate nand|mux] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one bootstrapped gate (default gate_nand) over a batch of B ciphertexts per GPU on synthetic data:
seeded keys in the reference's RNG order, uniformly random LWE samples as operands (the bootstrap does the same work
whatever the plaintexts are).  B defaults to 4096 on one GPU (BASELINE.json configs[1]) and to 8192 per GPU under
torchrun (configs[4]: 65536 ciphertexts over 8 GPUs).  n=500, N=1024, k=1, l=2, Bg=2^10, key switch t=8 base 4.

  value          gates/s, whole job, operands resident in HBM when the timed region starts
  e2e            the same gate through the public API (vm.gate_nand) with HOST operands: pinned host -> device copies
                 and the device -> host read of the result are inside the timed region
  roofline       the blind-rotate kernel against the measured HBM peak (MEASURED_PEAKS.json), bytes per SURVEY.md
                 section 8(d)'s per-step model: n * (16384 * B + 65536) per launch -- the roofline BASELINE.json judges
  roofline_issue the same launch against what actually binds it: warp-instruction issue slots (static SASS count of
                 the build x the work of the launch, against SMs x 4 schedulers x the SM clock sampled in the run)
  mux, ntt       the other two legs of BASELINE.json's metric, measured in the same process (N = 1 only):
                 gate_mux at the same batch, and the stand-alone transform in GB/s against the HBM peak
  batch_sweep    gate_nand at {1, 16, 64, 256, 1024, 4096, 16384, 65536} ciphertexts on one GPU (BASELINE.json configs[3])
  per_gpu_batch_sweep   ms/gate at {256, 4096, 8192} ciphertexts per GPU (multi-GPU runs)
  parity_checked        the first outputs of the timed gate on EVERY rank against the CPU oracle, in the run
  cpu_baseline   the CPU port of the reference algorithm (oracle/, C + OpenMP) on a bounded sample, all host cores;
                 `c0_reference_closures` next to it is the reference's own NumPy closures (nufhe/*_cpu.py), which
                 need /root/reference and therefore only run in the build container (tools/c0_baseline.py)

`--impl reference` times the CPU port alone (the reference is pure Python + JIT-compiled Reikna kernels that cannot
run here; its algorithm is restated in oracle/ and pinned to its own closures, tests/golden/).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POLY = 1024
LWE_N = 500
SEED = 20260923
THREADS_PER_CT = 128            # throughput shape of the fused kernel: 2 ciphertexts on 256 threads


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=0, help='ciphertexts per GPU per step (0: 4096 on one GPU, 8192 per '
                                                         'GPU under torchrun)')
    ap.add_argument('--gate', default='nand', choices=['nand', 'mux'])
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--cpu-sample', type=int, default=0, help='gates in the CPU sample (0 = auto)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the mux / ntt / sweep legs (headline line only)')
    ap.add_argument('--ntt-transforms', type=int, default=262144)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the ciphertexts the last one returned (a, b, current_variances; '
                         'rank 0 under torchrun) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl b200)')
    return args


def host_cores():
    """Usable host threads: CPU affinity, capped by a cgroup CPU quota if the container has one."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def measured_peak_hbm():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


def lib_sha():
    from nufhe_b200 import _native
    with open(_native.LIB_PATH, 'rb') as f:
        return hashlib.sha256(f.read()).hexdigest()[:16]


def measured_traffic(batch, counts=None):
    """dram__bytes_read + dram__bytes_write of one blind-rotate launch from the committed ncu capture of this round
    (profiles/r2_traffic.json, written by tools/ncu_traffic.py from an ncu run of tools/profile_target.py; a profiler
    cannot run inside the bench).  The capture carries the hash of the library it was taken on and the static SASS
    instruction counts of its step loop; the provenance says whether the library of THIS run is the same file, or at
    least the same kernel code (same per-phase counts -- e.g. rebuilt after a comment changed the line info).
    Returns (bytes or None, provenance)."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'r2_traffic.json')) as f:
            d = json.load(f)
        if int(d['batch']) != int(batch):
            return None, 'profiles/r2_traffic.json was captured at batch %s' % d['batch']
        k = d['blind_rotate_kernel']
        fp = d.get('kernel_fingerprint')
        if d.get('lib_sha') == lib_sha():
            which = 'this build'
        elif counts and fp and fp.get('phases') == counts.get('phases'):
            which = 'same kernel code as this build: identical static instruction counts per phase'
        else:
            which = 'an earlier r2 build'
        return (int(k['dram_bytes_read']) + int(k['dram_bytes_write']),
                'ncu capture profiles/r2_traffic.json (%s)' % which)
    except Exception as e:
        return None, 'no capture (%s)' % type(e).__name__


def static_instruction_counts():
    """Per-thread, per-step SASS instruction counts of the fused kernel in the library this run loads
    (tools/sass_stats.py: nvdisasm on the .so, no GPU involved); the committed copy is the fallback."""
    from nufhe_b200 import _native
    try:
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'sass_stats.py'), '--json', '--lib',
                              _native.LIB_PATH], capture_output=True, text=True, timeout=240)
        d = json.loads(out.stdout.strip().splitlines()[-1])
        d['source'] = 'tools/sass_stats.py on the loaded library'
        return d
    except Exception:
        try:
            with open(os.path.join(ROOT, 'profiles', 'r2_sass_stats.json')) as f:
                d = json.load(f)
            d['source'] = 'profiles/r2_sass_stats.json (committed)'
            return d
        except Exception:
            return None


def c0_committed():
    try:
        with open(os.path.join(ROOT, 'profiles', 'r2_c0_reference_closures.json')) as f:
            return json.load(f)
    except Exception:
        return {'available': False, 'why': 'the reference closures need /root/reference (build container only); '
                                           'run tools/c0_baseline.py there'}


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(directory, a, b, current_variances):
    """Write one step's destination ciphertexts (host arrays) as DIR/<name>.npy.  The int32 torus values go out as
    float64, which holds every one exactly.  When all ciphertexts would exceed DUMP_LIMIT_BYTES, a fixed seeded
    sample of them is written instead, with their indices in rows.npy."""
    import numpy
    n = b.shape[0]
    per_ct = 8 * a.shape[-1] + 8 + 4 + 8          # a, b, current_variances and the index of a sampled ciphertext
    arrays = {'a': a.astype(numpy.float64), 'b': b.astype(numpy.float64),
              'current_variances': current_variances.astype(numpy.float32)}
    if n * per_ct > DUMP_LIMIT_BYTES:
        keep = (DUMP_LIMIT_BYTES - 4096) // per_ct    # 4096: room for the .npy headers
        rows = numpy.sort(numpy.random.RandomState(SEED).choice(n, keep, replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays['rows'] = rows.astype(numpy.float64)
    os.makedirs(directory, exist_ok=True)
    for name, arr in arrays.items():
        numpy.save(os.path.join(directory, name + '.npy'), arr)


def metric_name(args):
    return 'bootstrapped gates/sec (%s) at batch %d per GPU' % (args.gate.upper(), args.batch)


def workload_name(args):
    return ('gate_%s batch=%d/GPU, NTT transform, n=500 N=1024 k=1 l=2 Bg=2^10, keyswitch t=8 base=4, '
            'seeded keys (reference RNG order), uniform random LWE operands' % (args.gate, args.batch))


# --------------------------------------------------------------------------- CPU arm

def oracle_keys():
    from oracle import oracle as O
    if oracle_keys.keys is None:
        oracle_keys.keys = O.OracleKeys(SEED)
    return oracle_keys.keys


oracle_keys.keys = None


def cpu_gate_sample(sample, gate):
    """Time the CPU oracle port on `sample` gates with all host threads.  Returns gates/s."""
    import numpy
    from oracle import oracle as O
    O.set_threads(host_cores())
    keys = oracle_keys()
    rng = numpy.random.RandomState(1)
    ops = [(rng.randint(-2**31, 2**31, size=(sample, LWE_N), dtype=numpy.int32),
            rng.randint(-2**31, 2**31, size=(sample,), dtype=numpy.int32)) for _ in range(3)]
    t = time.perf_counter()
    if gate == 'nand':
        O.gate_binary('nand', ops[0], ops[1], keys.bk, keys.ks)
    else:
        O.gate_mux(ops[0], ops[1], ops[2], keys.bk, keys.ks)
    dt = time.perf_counter() - t
    return sample / dt, dt


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = host_cores()
    sample = args.cpu_sample or max(cores * 8, 16)
    for _ in range(args.warmup):
        cpu_gate_sample(min(sample, cores), args.gate)
    t_total = 0.0
    for _ in range(args.steps):
        _, dt = cpu_gate_sample(sample, args.gate)
        t_total += dt
    value = sample * args.steps / t_total
    line = {
        'impl': 'reference', 'metric': metric_name(args), 'value': value, 'unit': 'gates/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * t_total / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'u64', 'data': 'synthetic',
        'config': {'workload': workload_name(args),
                   'note': 'CPU PORT of the reference algorithm (oracle/nufhe_oracle.c, C + OpenMP, all host cores) '
                           '-- a generous stand-in: the reference\'s own NumPy closures run ~2500x slower per core '
                           '(c0_reference_closures).  Each step is a bounded sample of %d gates of the workload'
                           % sample},
        'cpu_baseline': {'value': value, 'unit': 'gates/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d gate_%s per step, %d steps' % (sample, args.gate, args.steps)},
        'c0_reference_closures': c0_committed(),
        'e2e': {'value': value, 'unit': 'gates/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- clocks sampler

class ClockSampler(threading.Thread):
    QUERY = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(
                    ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.QUERY,
                     '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(',')]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith('active') for s in self.samples)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': int(float(self.samples[0][1])), 'reasons': reasons,
                'samples': len(sm)}


# --------------------------------------------------------------------------- GPU arm

def run_b200_arm(args):
    import numpy
    import torch
    import torch.distributed as dist
    import nufhe_b200 as nufhe
    from nufhe_b200.lwe import LweSampleArray

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    ctx = nufhe.Context(rng=nufhe.DeterministicRNG(SEED), device_id=local_rank)
    thr = ctx.thread
    params = nufhe.NuFHEParameters()
    # Keys: rank 0 generates them (on its GPU, reference RNG order) and broadcasts the cloud key over
    # NCCL/NVLink once; there is no per-gate collective (SURVEY.md section 8e).
    if rank == 0:
        secret_key, cloud_key = ctx.make_key_pair()
    if world > 1:
        from nufhe_b200.api_low_level import NuFHECloudKey
        from nufhe_b200.bootstrap import BootstrapKey
        from nufhe_b200.tgsw import TransformedTGswSampleArray
        from nufhe_b200.lwe import LweKeyswitchKey
        if rank != 0:
            tg = TransformedTGswSampleArray.empty(thr, params.tgsw_params, (LWE_N,))
            ks_lwe = LweSampleArray.empty(thr, params.in_out_params, (N_POLY, 8, 4))
            cloud_key = NuFHECloudKey(params, BootstrapKey(params.in_out_params, tg), LweKeyswitchKey(ks_lwe))
        from nufhe_b200.sharding import cloud_key_tensors, broadcast_tensors
        broadcast_tensors(cloud_key_tensors(cloud_key), src=0)
        torch.cuda.synchronize()
    vm = ctx.make_virtual_machine(cloud_key)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=thr.device)   # > 126 MB L2
    launches_per_gate = 2          # fused bootstrap(s) + key switch, for NAND and for MUX alike

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps):
        """`steps` calls between two events on the launching stream, barrier + synchronize on both sides, max over ranks."""
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            step_fn()
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=thr.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    def make_case(B, gate_name, seed):
        """Operands (pinned host + device copies), destination and the two step functions for one (batch, gate)."""
        n_ops = 2 if gate_name == 'nand' else 3
        gen = torch.Generator(device='cpu').manual_seed(seed + rank)
        host_ops = []
        for _ in range(n_ops):
            a = torch.randint(-2**31, 2**31, (B, LWE_N), generator=gen, dtype=torch.int64).to(torch.int32).pin_memory()
            b = torch.randint(-2**31, 2**31, (B,), generator=gen, dtype=torch.int64).to(torch.int32).pin_memory()
            host_ops.append((a, b))
        dev_ops = [LweSampleArray(params.in_out_params, a.to(thr.device), b.to(thr.device),
                                  torch.zeros(B, dtype=torch.float32, device=thr.device)) for a, b in host_ops]
        dest = vm.empty_ciphertext((B,))
        gate = getattr(vm, 'gate_' + gate_name)
        out_host_a = torch.empty((B, LWE_N), dtype=torch.int32).pin_memory()
        out_host_b = torch.empty((B,), dtype=torch.int32).pin_memory()

        def device_step():
            flush_buf.fill_(1)                      # L2 flush, inside the timed region (~0.1 ms)
            gate(*dev_ops, dest=dest)

        def e2e_step():
            flush_buf.fill_(1)
            cts = [LweSampleArray(params.in_out_params, a.to(thr.device, non_blocking=True),
                                  b.to(thr.device, non_blocking=True),
                                  torch.zeros(B, dtype=torch.float32, device=thr.device)) for a, b in host_ops]
            r = gate(*cts)
            out_host_a.copy_(r.a, non_blocking=True)
            out_host_b.copy_(r.b, non_blocking=True)

        return dict(B=B, n_ops=n_ops, host_ops=host_ops, dev_ops=dev_ops, dest=dest, device_step=device_step,
                    e2e_step=e2e_step)

    def measure_case(case, steps, warmup, with_e2e=True):
        for _ in range(warmup):
            case['device_step']()
        ms = timed(case['device_step'], steps)
        out = {'ms_per_step': ms / steps, 'gates_per_s': world * case['B'] * steps / (ms * 1e-3),
               'ms_per_gate': ms / steps / (world * case['B'])}
        if with_e2e:
            for _ in range(max(1, warmup // 2)):
                case['e2e_step']()
            ms_e = timed(case['e2e_step'], steps)
            out['e2e_gates_per_s'] = world * case['B'] * steps / (ms_e * 1e-3)
            out['e2e_ms_per_step'] = ms_e / steps
        return out

    B = args.batch
    main = make_case(B, args.gate, 1234)
    for _ in range(args.warmup):
        main['device_step']()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_total = timed(main['device_step'], args.steps)
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        # now: the stand-alone key switch timed below writes into the same buffers
        dest = main['dest']
        dump_outputs(args.dump_outputs, dest.a.cpu().numpy(), dest.b.cpu().numpy(),
                     dest.current_variances.cpu().numpy())
    for _ in range(max(1, args.warmup // 2)):
        main['e2e_step']()
    ms_e2e = timed(main['e2e_step'], args.steps)

    # ---- in-run parity: the first outputs of the timed gate on THIS rank against the CPU oracle (the engine's
    # seeded keys are the oracle's: tests/test_gpu_api.py::test_seeded_keys_equal_reference_keys)
    n_check = 8
    parity_ok = None
    if not args.no_cpu_baseline:
        from oracle import oracle as O
        O.set_threads(host_cores())
        keys = oracle_keys()
        ops_np = [(a[:n_check].numpy().copy(), b[:n_check].numpy().copy()) for a, b in main['host_ops']]
        if args.gate == 'nand':
            want = O.gate_binary('nand', ops_np[0], ops_np[1], keys.bk, keys.ks)
        else:
            want = O.gate_mux(ops_np[0], ops_np[1], ops_np[2], keys.bk, keys.ks)
        got_a, got_b = main['dest'].a[:n_check].cpu().numpy(), main['dest'].b[:n_check].cpu().numpy()
        parity_ok = bool((got_a == want[0]).all() and (got_b == want[1]).all())
        if world > 1:
            t = torch.tensor([1 if parity_ok else 0], dtype=torch.int32, device=thr.device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            parity_ok = bool(int(t.item()))

    # ---- the dominant kernel alone (blind rotate + extract), CUDA events on the launching stream
    from nufhe_b200.tgsw import engine_format
    bk_int = engine_format(thr, cloud_key.bootstrap_key.tgsw)
    ext = (thr.empty((B, N_POLY), torch.int32), thr.empty((B,), torch.int32))
    x1 = (main['dev_ops'][0].a, main['dev_ops'][0].b)
    x2 = (main['dev_ops'][1].a, main['dev_ops'][1].b)

    def kernel_ms(fn):
        ts = []
        for i in range(args.warmup + args.steps):
            flush_buf.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                ts.append(e0.elapsed_time(e1))
        return sum(ts) / len(ts)

    br_avg_ms = kernel_ms(lambda: thr.bootstrap_extract(x1, x2, 2**29, -1, -1, 2**29, bk_int, out=ext))
    ks_arrays = cloud_key.keyswitch_key.device_arrays()
    ks_avg_ms = kernel_ms(lambda: thr.keyswitch(ks_arrays, ext, out=(main['dest'].a, main['dest'].b)))

    extras = {}
    if not args.no_extras:
        if world == 1:
            other = 'mux' if args.gate == 'nand' else 'nand'
            r = measure_case(make_case(B, other, 4321), max(2, args.steps // 2), max(3, args.warmup))
            extras[other] = {'gates_per_s': r['gates_per_s'], 'ms_per_step': r['ms_per_step'],
                             'e2e_gates_per_s': r['e2e_gates_per_s'], 'batch': B,
                             'note': 'gate_%s at the same batch, same process; two bootstraps + one key switch per MUX'
                                     % other}
            torch.cuda.empty_cache()
            extras['ntt'] = measure_ntt(thr, args.ntt_transforms, flush_buf, measured_peak_hbm()[0])
            # BASELINE.json configs[3]: batch sweep of gate_nand on one GPU (device-resident operands, L2 flushed)
            sweep = []
            for b in (1, 16, 64, 256, 1024, 4096, 16384, 65536):
                r = measure_case(make_case(b, 'nand', 77), 3 if b <= 4096 else 2, 3, with_e2e=False)
                sweep.append({'batch': b, 'ms_per_step': r['ms_per_step'], 'ms_per_gate': r['ms_per_gate'],
                              'gates_per_s': r['gates_per_s'],
                              'hbm_gbs_per_step_model': LWE_N * (16384 * b + 65536) / (r['ms_per_step'] * 1e-3) / 1e9})
                torch.cuda.empty_cache()
            extras['batch_sweep'] = sweep
        else:
            sweep = []
            for b in (256, 4096, 8192):
                r = measure_case(make_case(b, 'nand', 99), 3, 3, with_e2e=False)
                sweep.append({'per_gpu_batch': b, 'global_batch': world * b, 'ms_per_gate': r['ms_per_gate'],
                              'gates_per_s': r['gates_per_s']})
            extras['per_gpu_batch_sweep'] = sweep

    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        clocks = sampler.summary()
        alg_bytes = LWE_N * (16384 * B + 65536)
        achieved = alg_bytes / (br_avg_ms * 1e-3) / 1e9
        ms_per_step = ms_total / args.steps
        value = world * B * args.steps / (ms_total * 1e-3)
        e2e_value = world * B * args.steps / (ms_e2e * 1e-3)
        n_ops = main['n_ops']
        h2d = world * n_ops * (B * LWE_N * 4 + B * 4)     # whole job, all ranks
        d2h = world * (B * LWE_N * 4 + B * 4)
        counts = static_instruction_counts()
        traffic, traffic_src = measured_traffic(B, counts)
        line = {
            'metric': metric_name(args), 'value': value, 'unit': 'gates/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'u64', 'data': 'synthetic',
            'config': {'workload': workload_name(args), 'global_batch': world * B, 'per_gpu_batch': B,
                       'parallelism': 'ciphertext-sharded x%d, cloud key broadcast once over NCCL' % world,
                       'l2': 'flushed by a 256 MiB fill before every step (inside the timed region)',
                       'ms_per_gate': ms_per_step / (world * B),
                       'published_reference_ms_per_gate': 0.35,
                       'published_note': 'nufhe README.md:64-65, NTT path, unnamed GPU and batch; not the same '
                                         'hardware/config, so vs_baseline stays null'},
            'e2e': {'value': e2e_value, 'unit': 'gates/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'ms_per_step': ms_e2e / args.steps},
            'gpu_launches': launches_per_gate * args.steps,
            'clocks': clocks,
            'roofline': {'bound': 'hbm', 'kernel': 'blind_rotate_kernel', 'achieved': achieved, 'peak': peak,
                         'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic, 'traffic_source': traffic_src,
                         'algorithmic_bytes': alg_bytes,
                         'peak_source': peak_src, 'bytes_model': 'per-step: n*(16384*B+65536) per launch',
                         'ms_per_launch': br_avg_ms, 'share_of_step': br_avg_ms / ms_per_step,
                         'note': 'the roofline BASELINE.json names; the kernel is integer-issue bound '
                                 '(roofline_issue), its real DRAM traffic is `traffic`'},
            'kernels_ms': {'blind_rotate_extract': br_avg_ms, 'keyswitch': ks_avg_ms},
            'parity_checked': {'outputs_per_rank': n_check if parity_ok is not None else 0, 'ranks': world,
                               'ok': parity_ok, 'against': 'CPU oracle (oracle/), same seeded keys'},
            'build': thr.build_info(), 'lib_sha': lib_sha(),
        }
        if counts:
            per_thread = counts['per_thread_step_total']
            warp_instr = per_thread * LWE_N * B * THREADS_PER_CT / 32.0
            sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
            mhz = clocks.get('sm_mhz') or clocks.get('sm_max_mhz') or 1965
            peak_issue = sm_count * 4 * mhz * 1e6                       # warp-instructions per second
            ach = warp_instr / (br_avg_ms * 1e-3)
            alu = counts['per_thread_step']['alu']
            line['roofline_issue'] = {
                'bound': 'int_issue', 'kernel': 'blind_rotate_kernel',
                'warp_instructions_per_launch': warp_instr, 'achieved': ach / 1e9, 'peak': peak_issue / 1e9,
                'unit': 'G warp-instr/s', 'frac': ach / peak_issue,
                'instructions_per_thread_step': per_thread, 'alu_pipe_instructions_per_thread_step': alu,
                'alu_pipe_frac': (alu * LWE_N * B * THREADS_PER_CT / 32.0 * 2) / (br_avg_ms * 1e-3) / peak_issue,
                'peak_model': '%d SMs x 4 schedulers x %d MHz (median SM clock sampled in the timed region); the ALU '
                              'pipe takes 2 cycles per warp-instruction (tools/microbench/pipes.cu)' % (sm_count, mhz),
                'count_source': counts['source'],
                'note': 'static SASS count of the step loop x 500 steps x %d threads per ciphertext; prologue, '
                        'epilogue and the rare canonicalisation path are not counted' % THREADS_PER_CT}
        line.update(extras)
        if not args.no_cpu_baseline:
            cores = host_cores()
            sample = args.cpu_sample or max(cores * 40, 64)
            cpu_gate_sample(min(sample, cores), args.gate)
            v, dt = cpu_gate_sample(sample, args.gate)
            line['cpu_baseline'] = {'value': v, 'unit': 'gates/s', 'cores': cores, 'kind': 'port',
                                    'sample': '%d gate_%s, %.1f s wall, oracle/nufhe_oracle.c + OpenMP'
                                              % (sample, args.gate, dt)}
            line['c0_reference_closures'] = c0_committed()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def measure_ntt(thr, transforms, flush_buf, peak):
    """Stand-alone batched transform (nb_ntt_forward_i32 / nb_ntt_inverse_i32, natural order both sides):
    algorithmic bytes 12288 per transform (4096 in + 8192 out, SURVEY.md 8d) over the CUDA-event time."""
    import ctypes
    import torch
    gen = torch.Generator(device='cpu').manual_seed(5)
    polys = torch.randint(-2**31, 2**31, (transforms, N_POLY), generator=gen, dtype=torch.int64).to(torch.int32).to(thr.device)
    f = thr.ntt_forward_i32(polys)
    back = torch.empty_like(polys)

    def fwd():
        thr._call('nb_ntt_forward_i32', ctypes.c_void_p(polys.data_ptr()), ctypes.c_void_p(f.data_ptr()), transforms)

    def inv():
        thr._call('nb_ntt_inverse_i32', ctypes.c_void_p(f.data_ptr()), ctypes.c_void_p(back.data_ptr()), transforms)

    def med(fn):
        ts = []
        for i in range(8):
            flush_buf.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1))
        return sorted(ts)[len(ts) // 2]

    mf, mi = med(fwd), med(inv)
    ok = bool(torch.equal(back, polys))
    alg = transforms * 12288
    return {'transforms': transforms, 'bytes_per_transform': 12288, 'fwd_ms': mf, 'inv_ms': mi,
            'fwd_gbs': alg / mf / 1e6, 'inv_gbs': alg / mi / 1e6, 'fwd_hbm_frac': alg / mf / 1e6 / peak,
            'inv_hbm_frac': alg / mi / 1e6 / peak, 'roundtrip_exact': ok}


def main():
    args = parse_args()
    if not args.batch:
        args.batch = 4096 if int(os.environ.get('WORLD_SIZE', '1')) == 1 else 8192
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == '__main__':
    main()
