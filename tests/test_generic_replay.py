"""Emitted GENERIC kernels (the fallback for unaligned / strided / 1-D / index-dimension fields) replayed on the CPU
(tests/march_emulator.py::run_generic: the CUDA source compiled unchanged by g++, one call per CUDA thread over the grid
``psad_plan_launch`` chose) against the committed golden vectors of the reference's own assignments and the oracle."""
import numpy as np
import pytest

import march_emulator as emu
from golden_util import build_op, golden_arrays, golden_names
from oracle.evaluate import evaluate
from pystencils_autodiff_b200.emit import emit_generic


@pytest.mark.parametrize('name', golden_names())
def test_generic_kernels_against_reference_golden_vectors(name):
    for mode in (None, 'zeros'):
        op = build_op(name, mode)
        ins, outs, grads = golden_arrays(name, mode)
        shape = next(iter(ins.values())).shape
        for ir, gold in ((op.forward_ast_gpu, outs), (op.backward_ast_gpu, grads)):
            ek = emit_generic(ir)
            arrays, named = [], {}
            for f in ek.fields:
                a = np.full(shape, np.nan, dtype=f.dtype.numpy_dtype)
                if f in ir.input_fields:
                    a[...] = ins.get(f.name, 0.0)        # '+=' outputs (time-constant fields) start from zero
                arrays.append(a)
                named[f.name] = a
            emu.run_generic(ek, arrays)
            for f in ir.output_fields:
                scale = max(1.0, np.abs(gold[f.name]).max())
                assert np.abs(named[f.name] - gold[f.name]).max() <= 1e-12 * scale, (name, mode, f.name)


def test_generic_kernel_strided_views_and_launch_range():
    """Non-contiguous fields (a transposed view, a view with a pitch) and a launch range: cells outside the iteration
    range but inside the write range become 0, cells outside the write range are not touched."""
    import pystencils_autodiff_b200 as ps
    u, out = ps.fields('u, out: float64[9,14]')
    op = ps.AutoDiffOp([ps.Assignment(out.center, 0.5 * u[0, 0] + 0.25 * u[1, -2] - u[-1, 1] * u[0, 1])], op_name='strided',
                       boundary_handling='zeros')
    ek = emit_generic(op.forward_ast_gpu)
    rng = np.random.default_rng(1)
    ut = np.asfortranarray(rng.standard_normal((9, 14)))              # x is NOT the contiguous axis
    big = np.full((9, 20), np.nan)
    ot = big[:, 3:17]                                                 # row pitch 20
    assert not ut.flags['C_CONTIGUOUS'] and not ot.flags['C_CONTIGUOUS']
    emu.run_generic(ek, [ot, ut])
    ref = evaluate(op.forward_assignments, {'u': np.ascontiguousarray(ut)}, 'zeros')['out']
    np.testing.assert_allclose(ot, ref, rtol=0, atol=1e-14)
    assert np.isnan(big[:, :3]).all() and np.isnan(big[:, 17:]).all()
    ot2 = np.full((9, 14), np.nan)
    emu.run_generic(ek, [ot2, ut], launch_range=dict(iter_lo=[3, 2], iter_hi=[6, 14], write_lo=[2, 0], write_hi=[7, 14]))
    assert np.isnan(ot2[:2]).all() and np.isnan(ot2[7:]).all()
    assert np.all(ot2[2] == 0) and np.all(ot2[6] == 0) and np.all(ot2[3:6, :2] == 0)
    np.testing.assert_allclose(ot2[3:6, 2:], ref[3:6, 2:], rtol=0, atol=1e-14)


def test_generic_kernel_one_dimensional_and_index_dimension():
    import pystencils_autodiff_b200 as ps
    a, b = ps.fields('a, b: float32[37]')
    op = ps.AutoDiffOp([ps.Assignment(b.center, a[1] - 2 * a[0] + a[-1])], op_name='lap1d', boundary_handling='zeros')
    x = np.random.default_rng(2).standard_normal(37).astype(np.float32)
    for ir, src, dst, assigns in ((op.forward_ast_gpu, 'a', 'b', op.forward_assignments),
                                  (op.backward_ast_gpu, 'diffb', 'diffa', op.backward_assignments)):
        ek = emit_generic(ir)
        res = np.full(37, np.nan, dtype=np.float32)
        emu.run_generic(ek, [res, x])
        ref = evaluate(assigns, {src: x.astype(np.float64)}, 'zeros')[dst]
        np.testing.assert_allclose(res, ref, rtol=0, atol=2e-6)
    # vector output (index dimension, array-of-structures layout): the curl-like case of tests/test_tfmad.py:341-401
    u = ps.Field.create_fixed_size('u', (8, 10), index_dimensions=0, dtype=np.float64)
    c = ps.Field.create_fixed_size('c', (8, 10, 2), index_dimensions=1, dtype=np.float64)
    disc = ps.fd.Discretization2ndOrder(dx=1)
    op = ps.AutoDiffOp(ps.AssignmentCollection([ps.Assignment(c.center(0), disc(ps.fd.Diff(u, 0))),
                                                ps.Assignment(c.center(1), disc(ps.fd.Diff(u, 1)))], []),
                       op_name='curl', boundary_handling='zeros')
    ek = emit_generic(op.forward_ast_gpu)
    U = np.random.default_rng(3).standard_normal((8, 10))
    C = np.full((8, 10, 2), np.nan)
    emu.run_generic(ek, [C if f.name == 'c' else U for f in ek.fields])
    ref = evaluate(op.forward_assignments, {'u': U}, 'zeros')['c']
    np.testing.assert_allclose(C, ref, rtol=0, atol=1e-14)


@pytest.mark.parametrize('seed', range(24))
def test_random_stencils_generic_replay(seed):
    """Every random stencil of the GPU fuzz test (tests/test_gpu_fuzz.py) through the GENERIC kernels on the CPU: several
    inputs and outputs, offsets up to +-4, non-linear terms, both boundary modes, fp32 / fp64, 2-D / 3-D."""
    import pystencils_autodiff_b200 as ps
    from stencil_fuzz import random_stencil
    asg, bh, shape, dtype = random_stencil(seed)
    op = ps.AutoDiffOp(asg, boundary_handling=bh, op_name='fuzz%d' % seed)
    rng = np.random.default_rng(seed)
    tol = 2e-5 if dtype == 'float32' else 1e-11
    for collection, ir in ((op.forward_assignments, op.forward_ast_gpu), (op.backward_assignments, op.backward_ast_gpu)):
        ek = emit_generic(ir)
        arrays, named = [], {}
        for f in ek.fields:
            a = np.full(shape, np.nan, dtype=f.dtype.numpy_dtype)
            if f in ir.input_fields:
                a[...] = rng.uniform(-1, 1, size=shape)
            arrays.append(a)
            named[f.name] = a
        emu.run_generic(ek, arrays)
        ref = evaluate(collection, {f.name: named[f.name].copy() for f in ir.input_fields}, bh)
        assert all(np.count_nonzero(ref[f.name]) for f in ir.output_fields), (seed, 'empty interior')
        for f in ir.output_fields:
            scale = max(1.0, np.abs(ref[f.name]).max())
            assert np.isfinite(named[f.name]).all(), (seed, f.name)
            assert np.abs(named[f.name] - ref[f.name]).max() <= tol * scale, (seed, f.name)
