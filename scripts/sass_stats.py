"""Offline look at a kernel's machine code (no GPU needed): NVRTC -> cubin -> ``cuobjdump -sass``; prints registers,
the instruction mix of the whole kernel and of its hottest loop (the largest region closed by a backward branch that
contains the full-barrier wait of the consumer warps), and what that loop costs if every issue slot were used.

    python scripts/sass_stats.py c5            # forward + adjoint march kernels of a workload
    python scripts/sass_stats.py c3 x2         # the fused-pair kernel
    python scripts/sass_stats.py c3 float16    # the workload with float16 fields
    python scripts/sass_stats.py c3 bfloat16   # the workload with bfloat16 fields
For an issue-bound kernel (C5: sqrt / division chains) time ~ loop instructions x warp-steps / (SMs x 4 x clock)."""
import collections
import os
import re
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pystencils_autodiff_b200 import runtime  # noqa: E402
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel  # noqa: E402
from pystencils_autodiff_b200.configs import CONFIG_SHAPES, make_config  # noqa: E402

_INS = re.compile(r'^\s+/\*([0-9a-f]+)\*/\s+(@!?U?P\d+\s+)?([A-Z0-9_.]+)(.*?);')


def parse(sass):
    rows = []
    for line in sass.splitlines():
        m = _INS.match(line)
        if m:
            rows.append((int(m.group(1), 16), m.group(3), m.group(4)))
    return rows


_FP = ('FADD', 'FMUL', 'FFMA', 'DADD', 'DMUL', 'DFMA', 'MUFU')


def hottest_loop(rows):
    """(start, end) addresses of the consumers' step loop: the smallest region closed by a backward branch that holds
    (nearly) all of the kernel's floating-point instructions."""
    regions = []
    for addr, op, rest in rows:
        if op.startswith('BRA'):
            m = re.search(r'0x([0-9a-f]+)', rest)
            if m and int(m.group(1), 16) < addr:
                lo, hi = int(m.group(1), 16), addr
                fp = sum(1 for a, o, _ in rows if lo <= a <= hi and o.split('.')[0] in _FP)
                regions.append((fp, hi - lo, lo, hi))
    if not regions:
        return None
    top = max(r[0] for r in regions)
    fp, _, lo, hi = min((r for r in regions if r[0] >= 0.9 * top), key=lambda r: r[1])
    return (lo, hi) if fp else None


def report(ek, label, cells_per_step, cells):
    runtime.compile_source(ek.source, ek.cache_key, list(ek.options))
    path = runtime.cubin_path(ek.cache_key)
    sass = subprocess.check_output(['cuobjdump', '-sass', path]).decode()
    res = subprocess.check_output(['cuobjdump', '-res-usage', path]).decode()
    rows = parse(sass)
    mix = collections.Counter(op.split('.')[0] for _, op, _ in rows)
    print('%s  %s' % (label, ' '.join(re.findall(r'REG:\d+|STACK:\d+|SHARED:\d+', res))))
    print('  whole kernel: %d instructions  %s' % (len(rows), dict(mix.most_common(12))))
    ops = collections.Counter(op for _, op, _ in rows)
    tma = sum(v for k, v in ops.items() if k.startswith('UTMALDG'))
    syncs = sum(v for k, v in ops.items() if k.startswith('SYNCS'))
    local = sum(v for k, v in ops.items() if k.split('.')[0] in ('STL', 'LDL'))
    vec = {k: v for k, v in ops.items() if k.startswith(('LDS.128', 'STG.E.EF.128', 'STG.E.128', 'STS.128', 'LDG'))}
    print('  Blackwell markers: UTMALDG (TMA tensor loads) %d, SYNCS (mbarrier) %d, local-memory LDL/STL %d; vector memory ops %s'
          % (tma, syncs, local, vec))
    loop = hottest_loop(rows)
    if loop:
        body = [r for r in rows if loop[0] <= r[0] <= loop[1]]
        lm = collections.Counter(op.split('.')[0] for _, op, _ in body)
        fp = sum(v for k, v in lm.items() if k in _FP)
        steps = cells / cells_per_step          # warp-steps
        t = len(body) * steps / (148 * 4 * 1.965e9) * 1e3
        print('  step loop 0x%x-0x%x: %d instructions (%d FP/MUFU = %.1f per cell)  %s'
              % (loop[0], loop[1], len(body), fp, fp / (cells_per_step / 32), dict(lm.most_common(12))))
        print('  -> %.3f ms if every issue slot of 148 SMs x 4 schedulers at 1.965 GHz were used (static count: rarely '
              'taken blocks included)' % t)


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else 'c5'
    x2 = 'x2' in sys.argv[2:]
    dtype = next((a for a in sys.argv[2:] if a in ('float16', 'bfloat16', 'float32', 'float64')), None)
    op = make_config(name, dtype=dtype)
    cells = 1
    for s_ in CONFIG_SHAPES[name]['shape']:
        cells *= s_
    for which, ir in (('forward', op.forward_ast_gpu), ('adjoint', op.backward_ast_gpu)):
        k = CompiledKernel(ir)
        ek = k.emitted('march_x2') if x2 else k._emitted.get('march_nomask') or k._emitted['generic']
        g = getattr(ek, 'geometry', None) or {}
        # 3-D march kernels unroll the step body once per register-window phase: the loop holds NP steps
        np_ = (sum(g.get('HZ', (0, 0))) // (2 if x2 else 1) + 1) if g else 1
        per_step = 32 * g.get('RY', 1) * g.get('SX', 1) * np_ if g else 32
        report(ek, '%s %s (%s; loop = %d step%s)' % (name, which, ek.name, np_, 's' if np_ > 1 else ''), per_step, cells)


if __name__ == '__main__':
    main()
