"""GPU fuzz: random stencils (asymmetric halos, several fields / outputs, nonlinear terms, both boundary modes,
2-D / 3-D, fp32 / fp64), forward and adjoint kernels against the numpy oracle, every applicable variant."""
import numpy as np
import pytest

import pystencils_autodiff_b200 as ps
from oracle import evaluate
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
from stencil_fuzz import random_stencil

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('seed', range(24))
def test_random_stencil_matches_oracle(seed):
    import torch
    asg, bh, shape, dtype = random_stencil(seed)
    op = ps.AutoDiffOp(asg, boundary_handling=bh, op_name='fuzz%d' % seed)
    rng = np.random.default_rng(seed)
    tol = 2e-5 if dtype == 'float32' else 1e-11
    for collection, ir in ((op.forward_assignments, op.forward_ast_gpu), (op.backward_assignments, op.backward_ast_gpu)):
        k = CompiledKernel(ir)
        arrays = {f.name: rng.uniform(-1, 1, size=shape).astype(dtype) for f in ir.input_fields}
        ref = evaluate(collection, arrays, bh)
        assert all(np.count_nonzero(ref[f.name]) for f in ir.output_fields), (seed, 'empty interior')
        variants = ['generic'] + (['march'] if 'march' in k._emitted and shape[-1] * np.dtype(dtype).itemsize % 16 == 0 else [])
        for v in variants:
            tens = {n: torch.from_numpy(a).cuda() for n, a in arrays.items()}
            for f in ir.output_fields:
                tens[f.name] = torch.full(shape, float('nan'), dtype=getattr(torch, dtype), device='cuda')
            k(**{f.name: tens[f.name] for f in k.fields}, _variant=v)
            for f in ir.output_fields:
                got = tens[f.name].cpu().numpy()
                scale = max(1.0, np.abs(ref[f.name]).max())
                assert np.isfinite(got).all(), (seed, v, f.name)
                assert np.abs(got - ref[f.name]).max() <= tol * scale, (seed, v, f.name, np.abs(got - ref[f.name]).max())
