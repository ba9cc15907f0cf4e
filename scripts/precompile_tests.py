"""NVRTC-compile (no GPU needed) the kernels the golden-vector and slab time-loop GPU tests will ask for, into the in-tree
cubin cache that travels to the GPU box — so that the GPU suite spends its time running kernels, not compiling them.
    python scripts/precompile_tests.py"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from pystencils_autodiff_b200 import runtime  # noqa: E402
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel  # noqa: E402


def main():
    from golden_util import build_op, golden_names
    from pystencils_autodiff_b200.configs import heat3d_op, stencil27_op
    kernels = []
    for name in golden_names():
        for mode in (None, 'zeros'):
            op = build_op(name, mode)
            kernels += [CompiledKernel(op.forward_ast_gpu), CompiledKernel(op.backward_ast_gpu)]
    for make in (heat3d_op, stencil27_op):                      # tests/test_gpu_zz_slab_steps.py
        for bh in ('zeros', None):
            for shape in ((11, 30, 124), (15, 30, 124)):
                k = CompiledKernel(make(shape=shape, boundary_handling=bh).forward_ast_gpu)
                k.emitted('march_x2')
                kernels.append(k)
    from pystencils_autodiff_b200.configs import diffusion2d_op
    # tests/test_gpu_api.py time loops (fused pairs through the TimeLoop API), scripts/check_periodic.py (one rank and slabs
    # of two / four ranks, two ghost planes per side)
    for make, shapes in ((heat3d_op, ((24, 30, 128), (20, 30, 128), (28, 40, 256), (52, 40, 256), (100, 40, 256))),
                         (stencil27_op, ((20, 24, 128), (36, 24, 128), (68, 24, 128))),
                         (diffusion2d_op, ((64, 128),))):
        for shape in shapes:
            k = CompiledKernel(make(shape=shape).forward_ast_gpu)
            if k.fused_steps_reason() is None:
                k.emitted('march_x2')
            kernels.append(k)
    import pystencils_autodiff_b200 as ps
    from pystencils_autodiff_b200.configs import make_config
    from stencil_fuzz import random_stencil
    for seed in range(24):                                      # tests/test_gpu_fuzz.py
        asg, bh, shape, dtype = random_stencil(seed)
        op = ps.AutoDiffOp(asg, boundary_handling=bh, op_name='fuzz%d' % seed)
        kernels += [CompiledKernel(op.forward_ast_gpu), CompiledKernel(op.backward_ast_gpu)]
    import test_gpu_fuzz16 as f16                               # tests/test_gpu_fuzz16.py
    from stencil_fuzz import DOUBLE_SHAPES, fuzz_case
    cases = [fuzz_case(seed, dtype) for seed in range(24) for dtype in ('float16', 'bfloat16')]
    cases += [fuzz_case(seed, mixed=True) for seed in f16.MIXED_SEEDS]
    for dtype, seed in f16.DOUBLE_CASES:
        shape = DOUBLE_SHAPES[len(fuzz_case(seed, dtype)[3])]
        cases.append(fuzz_case(seed, dtype, shape=shape, data_type='double'))
    kernels += [CompiledKernel(ir) for case in cases for ir, _ in case[1]]
    import test_gpu_fuzz_pairs as fp                            # tests/test_gpu_fuzz_pairs.py: pairs of both row modes
    from stencil_fuzz import PAIR_SEEDS, pair_case
    pair_kernels = [fp.pair_kernel(ir, tuning) for seed in PAIR_SEEDS for _, ir, _ in pair_case(seed)[0]
                    for tuning in fp.ROW_MODES.values()]
    for seed in fp.SLAB_SEEDS:
        case, g = fp.slab_case(seed)
        pair_kernels += [CompiledKernel(case[0][0][1]), fp.slab_local_kernel(seed, g)]
    for k in pair_kernels:
        k.fused_steps_reason()                                  # emits the pair where it can be built
    kernels += pair_kernels
    for name, shape, dtype in (('c1', (20, 30), 'float32'), ('c1', (20, 32), 'float64'), ('c2', (96, 256), 'float32'),
                               ('c2', (33, 20), 'float64'), ('c3', (40, 48, 256), 'float32'), ('c4', (12, 20, 132), 'float64'),
                               ('c5', (3, 40, 136), 'float32')):       # tests/test_gpu_parity.py
        for bh in (None, 'zeros'):
            op = make_config(name, shape=shape, dtype=dtype, boundary_handling=bh)
            kernels += [CompiledKernel(op.forward_ast_gpu), CompiledKernel(op.backward_ast_gpu)]
    import sympy as sp                                          # tests/test_gpu_zz_golden.py: exact adjoint mode
    from pystencils_autodiff_b200.configs import tv_gradient_op
    x, y, z = ps.fields('x, y, z: float64[7,8]')
    asg = ps.AssignmentCollection({z.center: x[1, 0] * y[0, 0] + sp.sin(x[0, -1]) * y[-1, 1]})
    for mode in ('exact', 'reference'):
        for op in (ps.AutoDiffOp(asg, op_name='nl_' + mode, boundary_handling='zeros', adjoint_mode=mode),
                   tv_gradient_op(shape=(2, 6, 8), dtype='float64', adjoint_mode=mode)):
            kernels += [CompiledKernel(op.forward_ast_gpu), CompiledKernel(op.backward_ast_gpu)]
    t0 = time.time()
    hits = misses = 0
    for k in kernels:
        for v, ek in k._emitted.items():
            hit, _ = runtime.compile_source(ek.source, ek.cache_key, list(ek.options))
            hits += hit
            misses += not hit
    print('%d kernels: %d already cached, %d compiled in %.0f s' % (hits + misses, hits, misses, time.time() - t0))


if __name__ == '__main__':
    main()
