"""16-bit fields against the shipped precision, in one process on one GPU: forward and adjoint march kernels of C3, C2,
C5 (fp32) and the 27-point stencil C4 (fp64) at their BASELINE shapes, each in float16, in bfloat16 and in its own dtype,
alternated.

Every timed region is 20 launches of one kernel, started from an idle GPU (a pause before it, like bench.py's
cool-down: these B200s power-cap within ~150 ms of streaming), timed with CUDA events; the median over the repeats is
reported per launch, with the achieved bandwidth from ``StencilKernelIR.bytes_per_cell`` (compulsory HBM bytes).  The
accuracy of the 16-bit kernels is measured on sampled blocks against the fp64 oracle evaluated on the 16-bit inputs
converted exactly to fp64: max |got - ref| / max |ref| (DESIGN §6: <= 5e-4 for float16, <= 4e-3 for bfloat16).  Card
name, power limit and max SM clock are read in the same run.

Output per workload: ``speedup_forward`` / ``speedup_adjoint`` (float16 over the shipped dtype),
``speedup_bf16_forward`` / ``speedup_bf16_adjoint`` (bfloat16 over the shipped dtype) and ``bf16_over_fp16_forward`` /
``bf16_over_fp16_adjoint`` (float16 time / bfloat16 time: above 1 when bfloat16 is faster).

    python scripts/half_bench.py --out half_bench.json [--repeats 5] [--only c3,c4]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# workload -> (BASELINE shape, dtype it ships in)
WORKLOADS = {'c3': ((1024, 1024, 1024), 'float32'), 'c2': ((8192, 8192), 'float32'),
             'c5': ((16, 4096, 4096), 'float32'), 'c4': ((768, 768, 768), 'float64')}
LAUNCHES = 20


def card_info():
    import torch
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info['power_limit_and_max_sm_clock'] = q
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = 'not read: %s' % e
    return info


def make_inputs(op, shape, dtype, seed):
    import torch
    g = torch.Generator(device='cuda').manual_seed(seed)
    tens = {}
    for f in op.forward_input_fields:
        tens[f.name] = (torch.rand(shape, device='cuda', generator=g, dtype=torch.float32) + 0.5).to(dtype)
    return tens


def time_kernel(kernel, args, pause_s):
    import torch
    torch.cuda.synchronize()
    time.sleep(pause_s)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(LAUNCHES):
        kernel(**args)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / LAUNCHES


def sampled_error(name, shape, ir, tensors, which):
    """Max error over three blocks (corner, centre, far corner) relative to the largest reference value there."""
    from oracle import evaluate
    from pystencils_autodiff_b200.configs import make_config
    nd = len(shape)
    halo = [max(lo, hi) for lo, hi in ir.max_halo]
    block = {3: (12, 20, 128), 2: (64, 256)}[nd]
    block = tuple(min(b, s) for b, s in zip(block, shape))
    worst, scale = 0.0, 0.0
    for frac in (0.0, 0.5, 1.0):
        start = [int(frac * (s - b)) for s, b in zip(shape, block)]
        lo = [max(0, c - h) for c, h in zip(start, halo)]
        hi = [min(s, c + b + h) for c, b, s, h in zip(start, block, shape, halo)]
        sl = tuple(slice(a, b) for a, b in zip(lo, hi))
        inner = tuple(slice(c - a, c - a + b) for c, a, b in zip(start, lo, block))
        own = tuple(slice(c, c + b) for c, b in zip(start, block))
        ins = {f.name: tensors[f.name][sl].double().cpu().numpy() for f in ir.input_fields}
        op64 = make_config(name, shape=next(iter(ins.values())).shape, dtype='float64')
        assigns = op64.forward_assignments if which == 'forward' else op64.backward_assignments
        ref = evaluate(assigns, ins, 'zeros')
        for f in ir.output_fields:
            r = ref[f.name][inner]
            got = tensors[f.name][own].double().cpu().numpy()
            worst = max(worst, float(np.abs(got - r).max()))
            scale = max(scale, float(np.abs(r).max()))
    return worst / max(scale, 1e-30)


def run_workload(name, repeats, pause_s):
    import torch
    from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
    from pystencils_autodiff_b200.configs import make_config
    shape, base = WORKLOADS[name]
    cells = int(np.prod(shape))
    legs = {}
    dtypes = ('float16', 'bfloat16', base)
    for dt in dtypes:
        op = make_config(name, shape=shape, dtype=dt, boundary_handling='zeros')
        tdt = getattr(torch, dt)
        tens = make_inputs(op, shape, tdt, seed=1)
        fwd, bwd = CompiledKernel(op.forward_ast_gpu), CompiledKernel(op.backward_ast_gpu)
        for f in op.forward_output_fields:
            tens[f.name] = torch.empty(shape, dtype=tdt, device='cuda')
        for f in op.backward_ast_gpu.output_fields:
            tens[f.name] = torch.empty(shape, dtype=tdt, device='cuda')
        fargs = {f.name: tens[f.name] for f in fwd.fields}
        fwd(**fargs)                                  # warm-up (module load) and the adjoint's input
        for f in op.forward_output_fields:
            tens['diff' + f.name] = tens[f.name]
        bargs = {f.name: tens[f.name] for f in bwd.fields}
        bwd(**bargs)
        torch.cuda.synchronize()
        assert fwd.last_variant == 'march' and bwd.last_variant == 'march', (name, dt)
        legs[dt] = dict(op=op, fwd=fwd, bwd=bwd, fargs=fargs, bargs=bargs, tens=tens, ms_fwd=[], ms_bwd=[])
    for _ in range(repeats):
        for dt in dtypes:
            L = legs[dt]
            L['ms_fwd'].append(time_kernel(L['fwd'], L['fargs'], pause_s))
            L['ms_bwd'].append(time_kernel(L['bwd'], L['bargs'], pause_s))
    res = {'shape': list(shape), 'cells': cells, 'launches_per_region': LAUNCHES, 'repeats': repeats}
    for dt, L in legs.items():
        row = {}
        for which, ir, key in (('forward', L['op'].forward_ast_gpu, 'ms_fwd'), ('adjoint', L['op'].backward_ast_gpu, 'ms_bwd')):
            ms = float(np.median(L[key]))
            bpc = ir.bytes_per_cell()
            row[which] = {'ms_median': round(ms, 4), 'ms_all': [round(v, 4) for v in L[key]], 'bytes_per_cell': bpc,
                          'achieved_TBps': round(bpc * cells / (ms * 1e-3) / 1e12, 3),
                          'kernel': (L['fwd'] if which == 'forward' else L['bwd']).last_instance}
        if dt != base:
            # outputs of the last timed launches (inputs never change): checked on sampled blocks
            row['forward']['max_rel_err'] = sampled_error(name, shape, L['op'].forward_ast_gpu, L['tens'], 'forward')
            row['adjoint']['max_rel_err'] = sampled_error(name, shape, L['op'].backward_ast_gpu, L['tens'], 'backward')
        res[dt] = row
    for which in ('forward', 'adjoint'):
        ms = {dt: res[dt][which]['ms_median'] for dt in dtypes}
        res['speedup_' + which] = round(ms[base] / ms['float16'], 3)
        res['speedup_bf16_' + which] = round(ms[base] / ms['bfloat16'], 3)
        res['bf16_over_fp16_' + which] = round(ms['float16'] / ms['bfloat16'], 3)
    del legs
    torch.cuda.empty_cache()
    return res


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('--out', required=True)
    p.add_argument('--repeats', type=int, default=5)
    p.add_argument('--pause', type=float, default=0.5, help='idle seconds before every timed region')
    p.add_argument('--only', default=','.join(WORKLOADS))
    args = p.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('half_bench.py measures on a GPU; none is available')
    out = {'card': card_info(), 'workloads': {}}
    for name in args.only.split(','):
        out['workloads'][name] = run_workload(name, args.repeats, args.pause)
        print(json.dumps({name: out['workloads'][name]}), flush=True)
        with open(args.out, 'w') as fh:
            json.dump(out, fh, indent=1)
    out['card_after'] = card_info()
    with open(args.out, 'w') as fh:
        json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
