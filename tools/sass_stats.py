#!/usr/bin/env python
"""Static per-phase / per-pipe instruction counts of the fused bootstrap kernel, from the SASS of the built
library (no GPU needed).  The kernel is bound by the integer ALU pipe, so the ALU column of the step loop is
the number that predicts its run time; use this to judge an arithmetic change before spending GPU minutes.

    python tools/sass_stats.py [--kernel blind_rotate_kernel] [--by-func] [--lib path/to/lib.so]
    python tools/sass_stats.py --kernel blind_rotate_fft_kernel [--json]

The FP64 FFT kernel (--kernel blind_rotate_fft_kernel, or _ZN2nb23blind_rotate_fft_kernelINS_8BrFftCfgILi4E for the
4-ciphertext shape) gets its own report: FP64 instructions, the LDS / STS / LDG split and modelled shared-memory / L1
wavefronts per phase (fft_kernel_stats).  The default stays the NTT kernel: the committed DRAM-traffic capture
(profiles/r2_traffic.json) carries that kernel's per-phase counts as its fingerprint.

Each SASS instruction is attributed (through nvdisasm's inline chains, the library is built with -lineinfo)
to the line of `br2_step` in kernels.cuh that called it, i.e. to a phase.  Counts are static: fwd1 / fwd2 /
fwd3 are multiplied by their two sweeps per step (the `it` loops are not unrolled), the MAC by its two row
iterations, and code inside the warp-uniform `switch (g)` of fwd2 / inv2 counts a quarter -- see `per step`.
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ALU = ('IADD3', 'IADD', 'LOP3', 'SHF', 'SEL', 'ISETP', 'PRMT', 'VIADD', 'LEA', 'IMNMX', 'VIMNMX', 'MOV', 'PLOP3', 'P2R',
       'R2P', 'IABS', 'FLO', 'POPC', 'BREV', 'SGXT', 'BMSK', 'LOP', 'FSEL', 'FMNMX', 'CS2R', 'VABSDIFF', 'FSETP', 'I2FP')
FMA = ('IMAD', 'FFMA', 'FMUL', 'FADD', 'HFMA2', 'IDP')
LSU = ('LDS', 'STS', 'LDG', 'STG', 'LD', 'ST', 'LDSM', 'ATOMS', 'ATOMG', 'RED', 'LDC', 'LDCU', 'UBLKCP', 'SYNCS')
UNI = ('UMOV', 'UIADD3', 'ULEA', 'ULOP3', 'UISETP', 'USHF', 'UIMAD', 'S2UR', 'UPLOP3', 'USEL', 'UPRMT', 'R2UR', 'UFLO',
       'UP2UR', 'UIADD')


def pipe_of(op):
    base = op.split('.')[0]
    if base in ALU:
        return 'alu'
    if base in FMA:
        return 'fma'
    if base in LSU:
        return 'lsu'
    if base in UNI:
        return 'uni'
    return 'other'


COST = {'IMAD.WIDE(+R64)': 4, 'IMAD.WIDE(+RZ)': 4}
STEP_MULT = {'phase_fwd1': 2, 'phase_fwd2': 2, 'phase_fwd3': 2, 'phase_mac': 2}


def instruction_form(op, rest):
    """Opcode with the distinctions that matter for issue cost: carry-out predicates, 64-bit addends."""
    carry_out = bool(re.match(r'\s*R\w+, P\d', rest))
    if op.startswith('IMAD.WIDE'):
        key = 'IMAD.WIDE(+RZ)' if rest.rstrip(' ;').endswith('RZ') else 'IMAD.WIDE(+R64)'
    elif op.startswith('IADD3'):
        key = 'IADD3.X' if '.X' in op else 'IADD3'
    elif op.startswith('IMAD.HI'):
        key = 'IMAD.HI'
    else:
        key = re.sub(r'\.(LUT|U32|AND|OR|EX|GE|GT|LT|LE|NE|EQ|W|L|R|HI|64|128|E|CONSTANT|RECONVERGENT)\b', '', op)
    return key + ('.P' if carry_out and key.startswith(('IMAD', 'IADD3')) else '')


def enclosing_functions(path):
    """line -> name of the enclosing function (rough: last line that looks like a definition at depth <= 1)."""
    names = {}
    cur = None
    rx = re.compile(r'^\s*(?:template\s*<[^>]*>\s*)?(?:NB_HD|NB_D|NB_HDC|__global__|__device__)\b.*?\b([A-Za-z_][A-Za-z0-9_]*)\s*\(')
    try:
        with open(path) as f:
            for i, line in enumerate(f, 1):
                m = rx.match(line)
                if m:
                    cur = m.group(1)
                names[i] = cur
    except OSError:
        pass
    return names


FP64 = ('DFMA', 'DADD', 'DMUL')
FFT_PHASES = ('fwd1', 'fwd2', 'fwd3', 'mac', 'inv3', 'inv2', 'inv1')


def block_lines(src, start_pred):
    """Lines of the braced blocks that open on a line satisfying start_pred (the opening line included)."""
    out = set()
    for i, l in enumerate(src, 1):
        if start_pred(l):
            depth, j = 0, i
            while j <= len(src):
                depth += src[j - 1].count('{') - src[j - 1].count('}')
                out.add(j)
                if depth <= 0 and j > i:
                    break
                j += 1
    return out


def fft_kernel_stats(text, kernel):
    """Per-phase counts of the FP64 FFT kernel (blind_rotate_fft_kernel, fft_kernels.cuh): the phases are the br_fft.cuh
    calls of br_fft_step.  Per thread and step: fwd2 / fwd3 / inv3 / inv2 run two sweeps, the MAC 512 / THREADS points,
    and the digit loop of fwd1 and the limb loop of inv1 (br_fft.cuh) two iterations.  Shared-memory and L1 wavefronts
    are modelled per warp-instruction: a 16 B access per lane is 4 wavefronts, 8 B is 2, 4 B is 1; the tw2 reads of
    passes 2 / 3 touch 8 distinct entries per warp, 1 wavefront."""
    kpath = os.path.join(ROOT, 'nufhe_b200', 'csrc', 'fft_kernels.cuh')
    fpath = os.path.join(ROOT, 'nufhe_b200', 'csrc', 'br_fft.cuh')
    ksrc = open(kpath).read().splitlines()
    fsrc = open(fpath).read().splitlines()
    phase_lines, in_step = {}, False
    names = {'fft_step_fwd1': 'fwd1', 'fft_fwd2': 'fwd2', 'fft_fwd3': 'fwd3', 'fft_step_mac': 'mac',
             'fft_inv3': 'inv3', 'fft_inv2': 'inv2', 'fft_step_inv1': 'inv1'}
    for i, line in enumerate(ksrc, 1):
        if 'void br_fft_step' in line:
            in_step = True
        elif in_step:
            m = re.search(r'\b(fft_[a-z0-9_]+)(?:<[a-z]+>)?\(', line)
            if m and m.group(1) in names:
                phase_lines[i] = names[m.group(1)]
            if line.startswith('}'):
                in_step = False
    twice = block_lines(fsrc, lambda l: 'for (int j = 0; j < 2; j++)' in l or 'for (int limb = 0; limb < 2; limb++)' in l)
    tw2_lines = {i for i, l in enumerate(fsrc, 1) if 'tw2[' in l}
    ct = int(re.search(r'BrFftCfgILi(\d+)E', kernel).group(1)) if re.search(r'BrFftCfgILi(\d+)E', kernel) else 2
    mult = {'fwd1': 1, 'fwd2': 2, 'fwd3': 2, 'mac': 512 // (128 * ct), 'inv3': 2, 'inv2': 2, 'inv1': 1}
    rx_line = re.compile(r'//## File "([^"]+)", line (\d+)')
    rx_ins = re.compile(r'^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)(.*)')
    cols = ('fp64', 'alu', 'fma', 'lds', 'sts', 'ldg', 'other_lsu', 'uni', 'other', 'total', 'wavefronts')
    counts = {ph: collections.Counter() for ph in FFT_PHASES}
    in_kernel, chain, chain_done = False, [], False
    for ln in text:
        if ln.startswith('.text.'):
            in_kernel = kernel in ln
            chain = []
            continue
        if not in_kernel:
            continue
        m = rx_line.search(ln)
        if m:
            if not chain or chain_done:
                chain, chain_done = [], False
            chain.append((m.group(1), int(m.group(2))))
            continue
        m = rx_ins.match(ln)
        if not m:
            continue
        chain_done = True
        phase = next((phase_lines[line] for path, line in chain if path.endswith('fft_kernels.cuh') and line in phase_lines), None)
        if phase is None:
            continue
        w = mult[phase] * (2 if any(path.endswith('br_fft.cuh') and line in twice for path, line in chain) else 1)
        op = m.group(1)
        base = op.split('.')[0]
        c = counts[phase]
        c['total'] += w
        if base in FP64:
            c['fp64'] += w
        elif base in ('LDS', 'STS', 'LDG'):
            c[base.lower()] += w
            width = 16 if '.128' in op else 8 if '.64' in op else 4
            wf = width // 4 if width > 4 else 1
            if base == 'LDS' and any(path.endswith('br_fft.cuh') and line in tw2_lines for path, line in chain):
                wf = 1
            c['wavefronts'] += w * wf
        elif pipe_of(op) == 'lsu':
            c['other_lsu'] += w
        else:
            c[pipe_of(op)] += w
    tot = collections.Counter()
    for c in counts.values():
        tot.update(c)
    return {'kernel': kernel, 'ct_per_cta': ct, 'columns': cols,
            'phases_per_thread_step': {ph: {k: counts[ph][k] for k in cols} for ph in FFT_PHASES},
            'per_thread_step': {'fp64': tot['fp64'], 'alu': tot['alu'], 'fma': tot['fma'],
                                'lsu': tot['lds'] + tot['sts'] + tot['ldg'] + tot['other_lsu'], 'uni': tot['uni'],
                                'other': tot['other']},
            'per_thread_step_total': tot['total'],
            'shared_l1_wavefronts_per_warp_step': tot['wavefronts'],
            'phases': {ph: counts[ph]['total'] for ph in FFT_PHASES}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--lib', default=os.path.join(ROOT, 'nufhe_b200', 'csrc', 'libnufhe_b200.so'))
    ap.add_argument('--kernel', default='blind_rotate_kernelINS_5BrCfgILi2ELi256',
                    help='substring of the mangled kernel name (default: the 2-ciphertext shape; the wide shape is '
                         'blind_rotate_kernelINS_5BrCfgILi1ELi256)')
    ap.add_argument('--by-func', action='store_true', help='also split each phase by innermost ff.cuh / br_phases function')
    ap.add_argument('--opcodes', action='store_true', help='per-step histogram of instruction forms (carry-out variants split)')
    ap.add_argument('--json', action='store_true', help='print one JSON object with the per-step totals (used by bench.py)')
    args = ap.parse_args()

    tmp = tempfile.mkdtemp()
    subprocess.check_call(['cuobjdump', '-xelf', 'all', os.path.abspath(args.lib)], cwd=tmp, stdout=subprocess.DEVNULL)
    cubin = [f for f in os.listdir(tmp) if f.endswith('.cubin')][0]
    text = subprocess.run(['nvdisasm', '--print-line-info-inline', '-c', os.path.join(tmp, cubin)],
                          capture_output=True, text=True).stdout.splitlines()

    if 'fft_kernel' in args.kernel:
        import json
        d = fft_kernel_stats(text, args.kernel)
        if args.json:
            print(json.dumps(d))
            return 0
        cols = d['columns']
        print('%-22s' % 'phase (per thread-step)' + ''.join('%11s' % c for c in cols))
        for ph, c in d['phases_per_thread_step'].items():
            print('%-22s' % ph + ''.join('%11.0f' % c[k] for k in cols))
        tot = {k: sum(c[k] for c in d['phases_per_thread_step'].values()) for k in cols}
        print('%-22s' % 'step' + ''.join('%11.0f' % tot[k] for k in cols))
        return 0

    # phase = line of kernels.cuh inside br2_step
    kpath = os.path.join(ROOT, 'nufhe_b200', 'csrc', 'kernels.cuh')
    ksrc = open(kpath).read().splitlines()
    phase_lines = {}
    in_step = False
    for i, line in enumerate(ksrc, 1):
        if 'void br2_step' in line:
            in_step = True
        if in_step:
            m = re.search(r'(phase_[a-z0-9_]+)', line)
            if m:
                phase_lines[i] = m.group(1)
            if line.startswith('}'):
                in_step = False
    step_call_lines = [i for i, l in enumerate(ksrc, 1) if 'br2_step<true' in l and 'void' not in l]
    if 'pair' in args.kernel:
        # the pair shape (blind_rotate_pair_kernel): phases are the pair_* calls of its step loop.  Each pair_* wrapper
        # holds BOTH thread halves (`if (h) f<1>(...) else f<0>(...)`), so a thread executes about half of the static
        # count of a split phase; the MAC loops run twice (two rows per thread).
        phase_lines, in_kernel_src = {}, False
        for i, line in enumerate(ksrc, 1):
            if 'blind_rotate_pair_kernel(' in line:
                in_kernel_src = True
            if in_kernel_src:
                m = re.search(r'\b(pair_[a-z0-9_]+)(?:<[a-z]+>)?\(', line)
                if m:
                    phase_lines[i] = 'phase_' + m.group(1)
                if line.startswith('}'):
                    in_kernel_src = False
        step_call_lines = list(phase_lines)

    # lines of br_phases.cuh inside a `switch (g)` (warp-uniform 4-way): each branch runs for a quarter of the warps
    bpath = os.path.join(ROOT, 'nufhe_b200', 'csrc', 'br_phases.cuh')
    case_lines = {i for i, l in enumerate(open(bpath).read().splitlines(), 1) if re.match(r'\s*(case \d+|default):', l)}

    # lines of br_phases.cuh inside the digit loop of phase_fwd1_both_digits (a real loop, two iterations per step)
    twice_lines = set()
    bsrc0 = open(bpath).read().splitlines()
    for i, l in enumerate(bsrc0, 1):
        if 'for (int j = 0; j < 2; j++)' in l:
            depth, j = 0, i
            while True:
                depth += bsrc0[j - 1].count('{') - bsrc0[j - 1].count('}')
                twice_lines.add(j)
                if depth <= 0 and j > i:
                    break
                j += 1

    # lines of br_phases.cuh inside an `if (canon_needed(...)) { ... }` block: the rare path of the deferred
    # canonicalisation (taken with probability ~2^-28 per task) -- not part of the executed step
    rare_lines = set()
    bsrc = open(bpath).read().splitlines()
    for i, l in enumerate(bsrc, 1):
        if 'canon_needed(' in l and l.lstrip().startswith('if '):
            depth, j = 0, i
            while True:
                depth += bsrc[j - 1].count('{') - bsrc[j - 1].count('}')
                rare_lines.add(j)
                if depth <= 0 and j > i:
                    break
                if depth <= 0 and '{' not in bsrc[j - 1]:
                    rare_lines.add(j + 1)     # single-statement body on the next line
                    break
                j += 1
            rare_lines.discard(i)             # the test itself is executed

    fn_maps = {}

    def fn_of(path, line):
        if path not in fn_maps:
            fn_maps[path] = enclosing_functions(path)
        return fn_maps[path].get(line)

    in_kernel = False
    chain = []
    counts = collections.defaultdict(lambda: collections.Counter())
    byfunc = collections.defaultdict(lambda: collections.Counter())
    rx_line = re.compile(r'//## File "([^"]+)", line (\d+)')
    rx_ins = re.compile(r'^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)(.*)')
    forms = collections.Counter()
    for ln in text:
        if ln.startswith('.text.'):
            in_kernel = args.kernel in ln
            chain = []
            continue
        if not in_kernel:
            continue
        m = rx_line.search(ln)
        if m:
            if not chain or chain_done:
                chain = []
                chain_done = False
            chain.append((m.group(1), int(m.group(2))))
            continue
        m = rx_ins.match(ln)
        if not m:
            continue
        chain_done = True
        op = m.group(1)
        pipe = pipe_of(op)
        phase = 'other'
        in_loop = False
        for path, line in chain:
            if path.endswith('kernels.cuh'):
                if line in phase_lines:
                    phase = phase_lines[line]
                if line in step_call_lines:
                    in_loop = True
        if phase != 'other' and not in_loop:
            phase = 'plain:' + phase     # the non-rotating instantiation (nb_external_product)
        w = 0.25 if any(path.endswith('br_phases.cuh') and line in case_lines for path, line in chain) else 1
        if any(path.endswith('br_phases.cuh') and line in twice_lines for path, line in chain):
            w *= 2
        if any(path.endswith('br_phases.cuh') and line in rare_lines for path, line in chain):
            counts['rare:' + phase][pipe] += w
            continue
        counts[phase][pipe] += w
        if args.opcodes and phase.startswith('phase_'):
            forms[instruction_form(op, m.group(2))] += w * (
                1 if ('BrCfgILi1E' in args.kernel and phase.startswith('phase_fwd')) else STEP_MULT.get(phase, 1))
        if args.by_func and chain:
            inner = None
            for path, line in chain:
                f = fn_of(path, line)
                if f and (path.endswith('ff.cuh')):
                    inner = f
                    break
            if inner is None:
                inner = fn_of(*chain[0]) or '?'
            byfunc[phase][(inner, pipe)] += w

    # the wide shape (1 ciphertext on 256 threads) runs the forward phases in one sweep
    mult = dict(STEP_MULT, phase_fwd1=1, phase_fwd2=1, phase_fwd3=1) if 'BrCfgILi1E' in args.kernel else STEP_MULT
    if args.json:
        import json
        tot = collections.Counter()
        for phase, c in counts.items():
            if phase.startswith('phase_'):
                for k, v in c.items():
                    tot[k] += v * mult.get(phase, 1)
        print(json.dumps({'kernel': args.kernel, 'per_thread_step': {k: tot[k] for k in ('alu', 'fma', 'lsu', 'uni', 'other')},
                          'per_thread_step_total': sum(tot.values()),
                          'phases': {ph: sum(c.values()) * mult.get(ph, 1) for ph, c in counts.items() if ph.startswith('phase_')}}))
        return 0
    print('%-22s %7s %7s %7s %7s %7s %8s' % ('phase (static)', 'alu', 'fma', 'lsu', 'uni', 'other', 'total'))
    tot = collections.Counter()
    for phase in sorted(counts):
        c = counts[phase]
        print('%-22s %7d %7d %7d %7d %7d %8d' % (phase, c['alu'], c['fma'], c['lsu'], c['uni'], c['other'], sum(c.values())))
        if phase.startswith('phase_'):
            for k, v in c.items():
                tot[k] += v * mult.get(phase, 1)
    print('%-22s %7d %7d %7d %7d %7d %8d   (sweeps, MAC rows and switch weights applied)' % (
        'per step, per thread', tot['alu'], tot['fma'], tot['lsu'], tot['uni'], tot['other'], sum(tot.values())))
    if args.opcodes:
        # issue cost in SMSP cycles per warp-instruction (tools/microbench/pipes.cu on B200): 2 on either integer
        # pipe, except IMAD.WIDE with a 64-bit addend: 4
        alu_c = sum(2 * v for k, v in forms.items() if pipe_of(k.split('(')[0]) == 'alu')
        fma_c = sum((COST.get(k.replace('.P', ''), 2)) * v for k, v in forms.items() if pipe_of(k.split('(')[0]) == 'fma')
        print('-- pipe cycles per step, per warp: ALU %.0f  FMA %.0f  (sum %.0f, balanced bound %.0f)' % (
            alu_c, fma_c, alu_c + fma_c, (alu_c + fma_c) / 2))
        print('-- instruction forms per step, per thread')
        for k, v in sorted(forms.items(), key=lambda kv: -kv[1]):
            if v >= 4:
                print('   %-20s %7.0f' % (k, v))
    if args.by_func:
        for phase in sorted(byfunc):
            if not phase.startswith('phase_'):
                continue
            print('--', phase)
            agg = collections.defaultdict(collections.Counter)
            for (fn, pipe), v in byfunc[phase].items():
                agg[fn][pipe] += v
            for fn, c in sorted(agg.items(), key=lambda kv: -sum(kv[1].values())):
                print('   %-24s alu %6d  fma %6d  lsu %5d  other %5d' % (fn, c['alu'], c['fma'], c['lsu'], c['uni'] + c['other']))


if __name__ == '__main__':
    sys.exit(main())
