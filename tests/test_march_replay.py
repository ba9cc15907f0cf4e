"""Emitted march kernels replayed on the CPU (tests/march_emulator.py): the per-step bodies — register-window slot
rotation, shuffled halos, plane sums, masks, vector stores, and the two-stage fused-step bodies of emit_chain.py —
run unchanged under g++ and are compared with the oracle.  TMA / mbarrier behaviour is covered by the GPU tests."""
import numpy as np
import pytest

import march_emulator as emu
from oracle.evaluate import evaluate
from pystencils_autodiff_b200 import configs
from pystencils_autodiff_b200.emit import MarchTuning, emit_march
from pystencils_autodiff_b200.emit_chain import chain_ineligible_reason, emit_march_chain


def _fields(ek, ir, shape, seed=0):
    rng = np.random.default_rng(seed)
    arrays, named = [], {}
    for f in ek.fields:
        a = emu.aligned_empty(shape, f.dtype.numpy_dtype)
        a[...] = rng.standard_normal(shape) if f in ir.input_fields else np.nan
        arrays.append(a)
        named[f.name] = a
    return arrays, named


@pytest.mark.parametrize('make, shape, bh, which, masked, tol', [
    (configs.heat3d_op, (5, 34, 132), 'zeros', 'forward', True, 3e-7),
    (configs.heat3d_op, (5, 34, 132), None, 'backward', True, 3e-7),
    (configs.heat3d_op, (5, 64, 256), 'zeros', 'forward', False, 3e-7),
    (configs.stencil27_op, (6, 30, 136), 'zeros', 'forward', True, 1e-14),
    (configs.stencil27_op, (6, 30, 136), None, 'backward', True, 1e-14),
    (configs.diffusion2d_op, (40, 260), 'zeros', 'forward', True, 3e-7),
])
def test_single_step_kernels_replay(make, shape, bh, which, masked, tol):
    op = make(shape=shape, boundary_handling=bh)
    ir = op.forward_ast_gpu if which == 'forward' else op.backward_ast_gpu
    assigns = op.forward_assignments if which == 'forward' else op.backward_assignments
    ek = emit_march(ir, None, masked=masked)
    arrays, named = _fields(ek, ir, shape)
    assert emu.run(ek, arrays) > 0
    ref = evaluate(assigns, {f.name: named[f.name].copy() for f in ir.input_fields}, boundary_handling=bh)
    for f in ir.output_fields:
        assert not np.isnan(named[f.name]).any()
        np.testing.assert_allclose(named[f.name], ref[f.name], rtol=0, atol=tol)


def _twice(assigns, fin, fout, u, bh):
    r1 = evaluate(assigns, {fin: u}, boundary_handling=bh)[fout].astype(u.dtype)
    return evaluate(assigns, {fin: r1}, boundary_handling=bh)[fout]


@pytest.mark.parametrize('make, shape, bh, which, tuning, tol', [
    (configs.heat3d_op, (5, 47, 124), 'zeros', 'forward', None, 4e-7),       # default fp32: rows exchanged between warps
    (configs.heat3d_op, (7, 23, 252), None, 'backward', MarchTuning(ry=2, ty=10, sx=4), 4e-7),
    (configs.heat3d_op, (5, 31, 124), 'zeros', 'forward', MarchTuning(exchange=False, ry=2, ty=30), 4e-7),   # rows recomputed
    (configs.heat3d_op, (5, 20, 132), None, 'forward', MarchTuning(exchange=False, ry=3, ty=9, sx=4), 4e-7),
    (configs.stencil27_op, (5, 17, 124), 'zeros', 'backward', MarchTuning(exchange=True, ry=3, ty=9, sx=4), 1e-14),
    (configs.stencil27_op, (5, 23, 68), 'zeros', 'forward', None, 1e-14),
    (configs.stencil27_op, (6, 17, 124), None, 'backward', MarchTuning(ry=2, ty=14, sx=4), 1e-14),
])
def test_fused_two_steps_replay(make, shape, bh, which, tuning, tol):
    """out = S(S(u)) from one launch == the oracle applied twice, including the zero border of the intermediate
    field (boundary None) and the zero reads outside the array ('zeros')."""
    op = make(shape=shape, boundary_handling=bh)
    ir = op.forward_ast_gpu if which == 'forward' else op.backward_ast_gpu
    assigns = op.forward_assignments if which == 'forward' else op.backward_assignments
    assert chain_ineligible_reason(ir) is None
    ek = emit_march_chain(ir, tuning)
    assert ek.plan['fused_steps'] == 2 and ek.plan['tile_x'] < ek.geometry['TX']
    assert (ek.plan['tile_y'] < ek.geometry['TY']) == ek.geometry['exchange'] == ('psad_consumer_barrier' in ek.source)
    arrays, named = _fields(ek, ir, shape, seed=3)
    assert emu.run(ek, arrays) > 0
    fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
    ref = _twice(assigns, fin, fout, named[fin].copy(), bh)
    assert not np.isnan(named[fout]).any()
    np.testing.assert_allclose(named[fout], ref, rtol=0, atol=tol)


def test_fused_steps_asymmetric_stencil_replay():
    """One-sided offsets in every direction (halo (1,0) / (0,1) / (1,0)): tile overlap and the accumulator rotation
    must follow the actual halo, not a symmetric radius."""
    import sympy as sp
    import pystencils_autodiff_b200 as ps
    shape = (6, 19, 124)
    u, out = ps.fields('u, out: float64[%d,%d,%d]' % shape)
    rhs = 0.5 * u[0, 0, 0] + 0.25 * u[-1, 0, 0] - 0.125 * u[0, 1, 0] + 0.0625 * u[0, 0, -1] + sp.Rational(1, 3) * u[0, 1, -1]
    op = ps.AutoDiffOp(ps.AssignmentCollection([ps.Assignment(out.center, rhs)]), op_name='skew', boundary_handling='zeros')
    for ir, assigns in ((op.forward_ast_gpu, op.forward_assignments), (op.backward_ast_gpu, op.backward_assignments)):
        assert chain_ineligible_reason(ir) is None
        ek = emit_march_chain(ir)
        arrays, named = _fields(ek, ir, shape, seed=5)
        emu.run(ek, arrays)
        fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
        ref = _twice(assigns, fin, fout, named[fin].copy(), 'zeros')
        np.testing.assert_allclose(named[fout], ref, rtol=0, atol=1e-14)


def test_fused_steps_eligibility():
    assert 'one input' in chain_ineligible_reason(configs.tv_gradient_op(shape=(2, 16, 32)).forward_ast_gpu)
    assert '3-D' in chain_ineligible_reason(configs.diffusion2d_op(shape=(16, 32)).forward_ast_gpu)
    with pytest.raises(ValueError):
        emit_march_chain(configs.diffusion2d_op(shape=(16, 32)).forward_ast_gpu)


@pytest.mark.parametrize('which', ['forward', 'backward'])
def test_tv_gradient_cross_cell_cse_replay(which):
    """Non-linear stencil with subexpressions: by default one CSE runs over all cells of a thread (shared gradient
    norms / reciprocal roots); must agree with the per-cell evaluation and with the oracle."""
    shape = (2, 33, 132)
    op = configs.tv_gradient_op(shape=shape)
    ir = op.forward_ast_gpu if which == 'forward' else op.backward_ast_gpu
    assigns = op.forward_assignments if which == 'forward' else op.backward_assignments
    results = []
    for cc in (None, False):
        ek = emit_march(ir, MarchTuning(cross_cse=cc), masked=True)
        assert ('const CT cs0' in ek.source) == (cc is None)
        rng = np.random.default_rng(0)
        arrays, named = [], {}
        for f in ek.fields:
            a = emu.aligned_empty(shape, f.dtype.numpy_dtype)
            a[...] = rng.random(shape) if f in ir.input_fields else np.nan
            arrays.append(a)
            named[f.name] = a
        emu.run(ek, arrays)
        results.append({f.name: named[f.name].copy() for f in ir.output_fields})
    ref = evaluate(assigns, {f.name: named[f.name].copy() for f in ir.input_fields}, boundary_handling='zeros')
    for f in ir.output_fields:
        scale = max(1.0, np.abs(ref[f.name]).max())
        for res in results:
            assert np.abs(res[f.name] - ref[f.name]).max() <= 2e-6 * scale


@pytest.mark.parametrize('seed', [0, 1, 2, 3, 5, 6])
def test_random_stencils_replay(seed):
    """The random stencils of the GPU fuzz test (asymmetric halos, several fields and outputs, non-linear terms, both
    boundary modes, 2-D / 3-D, fp32 / fp64), march variant, on the CPU."""
    import pystencils_autodiff_b200 as ps
    from stencil_fuzz import random_stencil
    from pystencils_autodiff_b200.emit import march_ineligible_reason
    asg, bh, shape, dtype = random_stencil(seed)
    if shape[-1] * np.dtype(dtype).itemsize % 16:
        pytest.skip('rows not 16-byte aligned: generic kernel only')
    op = ps.AutoDiffOp(asg, boundary_handling=bh, op_name='fuzz%d' % seed)
    rng = np.random.default_rng(seed)
    tol = 2e-5 if dtype == 'float32' else 1e-11
    for collection, ir in ((op.forward_assignments, op.forward_ast_gpu), (op.backward_assignments, op.backward_ast_gpu)):
        if march_ineligible_reason(ir):
            continue
        try:
            ek = emit_march(ir, None, masked=True)
        except ValueError:
            continue
        arrays, named = [], {}
        for f in ek.fields:
            a = emu.aligned_empty(shape, f.dtype.numpy_dtype)
            a[...] = rng.uniform(-1, 1, size=shape) if f in ir.input_fields else np.nan
            arrays.append(a)
            named[f.name] = a
        emu.run(ek, arrays)
        ref = evaluate(collection, {f.name: named[f.name].copy() for f in ir.input_fields}, bh)
        assert all(np.count_nonzero(ref[f.name]) for f in ir.output_fields), (seed, 'empty interior')
        for f in ir.output_fields:
            scale = max(1.0, np.abs(ref[f.name]).max())
            assert np.isfinite(named[f.name]).all(), (seed, f.name)
            assert np.abs(named[f.name] - ref[f.name]).max() <= tol * scale, (seed, f.name)


@pytest.mark.parametrize('bh, world', [('zeros', 2), (None, 3)])
def test_slab_launch_ranges_replay(bh, world):
    """The slab decomposition on the CPU: every rank's interior / boundary-plane launches (datahandling.slab_ranges)
    over its slab with ghost planes reproduce the unsharded launch bit for bit."""
    from pystencils_autodiff_b200.datahandling import slab_ranges
    shape = (6 if world == 2 else 9, 10, 132)
    op = configs.heat3d_op(shape=shape, boundary_handling=bh)
    ir = op.forward_ast_gpu
    g = 1
    rng = np.random.default_rng(11)
    u = emu.aligned_empty(shape, np.float32)
    u[...] = rng.standard_normal(shape)
    whole = emu.aligned_empty(shape, np.float32, np.nan)
    masked_kernel = emit_march(ir, None, masked=True)
    plain_kernel = emit_march(ir, None, masked=False)
    emu.run(plain_kernel if bh == 'zeros' else masked_kernel, [whole, u])
    ref = evaluate(op.forward_assignments, {'u': u.copy()}, boundary_handling=bh)['out']
    np.testing.assert_allclose(whole, ref, rtol=0, atol=3e-7)
    n = shape[0] // world
    for rank in range(world):
        start = rank * n
        local_u = emu.aligned_empty((n + 2 * g,) + shape[1:], np.float32, 0.0)
        lo, hi = max(0, start - g), min(shape[0], start + n + g)
        local_u[lo - (start - g):hi - (start - g)] = u[lo:hi]        # owned planes + received ghost planes
        local_out = emu.aligned_empty(local_u.shape, np.float32, np.nan)
        parts = slab_ranges(shape, start, n, g, rank > 0, rank < world - 1, 'zeros' if bh == 'zeros' else 'none',
                            ir.ghost_layers, 3)
        for part in parts:
            if part is None:
                continue
            same = part['iter_lo'] == part['write_lo'] and part['iter_hi'] == part['write_hi']
            emu.run(plain_kernel if same else masked_kernel, [local_out, local_u], launch_range=part)
        assert np.array_equal(local_out[g:g + n], whole[start:start + n]), rank


def test_replay_detects_a_missing_consumer_barrier():
    """The CTA-concurrent replay orders warps inside a step only through the kernel's own barrier: without it the
    neighbours' intermediate rows are read before they are written and the result is wrong."""
    shape = (5, 20, 124)
    op = configs.heat3d_op(shape=shape)
    ek = emit_march_chain(op.forward_ast_gpu, MarchTuning(exchange=True, ry=2, ty=8))
    assert ek.source.count('psad_consumer_barrier(cfg::THREADS);') == 3        # one per window phase
    ek.source = ek.source.replace('  psad_consumer_barrier(cfg::THREADS);\n', '')
    arrays, named = _fields(ek, op.forward_ast_gpu, shape, seed=0)
    emu.run(ek, arrays)
    ref = _twice(op.forward_assignments, 'u', 'out', named['u'].copy(), 'zeros')
    assert np.nanmax(np.abs(named['out'] - ref)) > 1e-3


def test_symbolic_scalar_and_fused_steps_replay():
    """A free scalar (alpha) reaches the kernels through the parameter block; with a symbolic coefficient the
    right-hand side only splits by z plane after expansion (emit_chain._planewise)."""
    import sympy as sp
    shape = (5, 12, 124)
    alpha = sp.Symbol('alpha')
    op = configs.heat3d_op(shape=shape, alpha=alpha)
    ir = op.forward_ast_gpu
    assert [s_.name for s_ in ir.scalars] == ['alpha']
    for ek, steps in ((emit_march(ir, None, masked=False), 1), (emit_march_chain(ir), 2),
                      (emit_march_chain(ir, MarchTuning(exchange=False)), 2)):
        arrays, named = _fields(ek, ir, shape, seed=4)
        emu.run(ek, arrays, scalars=[0.07])
        ref = named['u'].copy()
        for _ in range(steps):
            ref = evaluate(op.forward_assignments, {'u': ref}, boundary_handling='zeros', scalars={'alpha': 0.07})['out'].astype(np.float32)
        np.testing.assert_allclose(named['out'], ref, rtol=0, atol=5e-7)


def test_two_dimensional_interior_iteration_replay():
    """2-D march (row tiles instead of planes) with boundary None: zero border written by the kernel."""
    shape = (37, 132)
    op = configs.diffusion2d_op(shape=shape, boundary_handling=None)
    for ir, assigns in ((op.forward_ast_gpu, op.forward_assignments), (op.backward_ast_gpu, op.backward_assignments)):
        ek = emit_march(ir, None, masked=True)
        arrays, named = _fields(ek, ir, shape, seed=8)
        emu.run(ek, arrays)
        ref = evaluate(assigns, {f.name: named[f.name].copy() for f in ir.input_fields}, boundary_handling=None)
        for f in ir.output_fields:
            np.testing.assert_allclose(named[f.name], ref[f.name], rtol=0, atol=3e-7)
            assert (named[f.name][0] == 0).all() and (named[f.name][:, -1] == 0).all()


def test_fused_forward_adjoint_kernel_replay():
    """AutoDiffOp.fused_ast_gpu: forward and adjoint assignments of the README operator as one march kernel."""
    shape = (24, 64)
    op = configs.readme_op(shape=shape, boundary_handling='zeros')
    ir = op.fused_ast_gpu
    ek = emit_march(ir, None, masked=False)
    rng = np.random.default_rng(9)
    arrays, named = [], {}
    for f in ek.fields:
        a = emu.aligned_empty(shape, f.dtype.numpy_dtype)
        a[...] = rng.uniform(0.5, 1.5, size=shape) if f in ir.input_fields else np.nan
        arrays.append(a)
        named[f.name] = a
    emu.run(ek, arrays)
    fwd = evaluate(op.forward_assignments, {n: named[n].copy() for n in ('x', 'y')}, boundary_handling='zeros')
    bwd = evaluate(op.backward_assignments, {n: named[n].copy() for n in ('x', 'y', 'diffz')}, boundary_handling='zeros')
    np.testing.assert_allclose(named['z'], fwd['z'], rtol=2e-6, atol=1e-6)
    np.testing.assert_allclose(named['diffx'], bwd['diffx'], rtol=2e-6, atol=2e-6)
    np.testing.assert_allclose(named['diffy'], bwd['diffy'], rtol=2e-6, atol=2e-6)


# ---- the real march template (producer warp, TMA ring, full / empty mbarriers) on the CPU --------------------------------
@pytest.mark.timeout(300)
@pytest.mark.parametrize('make, shape, bh, tuning, chain, tol', [
    (configs.heat3d_op, (9, 12, 132), 'zeros', MarchTuning(ry=2, ty=6), False, 3e-7),            # register window, 5-slot ring
    (configs.heat3d_op, (7, 10, 132), None, MarchTuning(ry=1, ty=3, lookahead=1), False, 3e-7),  # shortest ring, masks
    (configs.stencil27_op, (6, 9, 68), 'zeros', MarchTuning(ry=3, ty=6, sx=4), False, 1e-14),     # arrival-time plane sums
    (configs.diffusion2d_op, (23, 132), 'zeros', MarchTuning(ry=1, ty=4), False, 3e-7),          # 2-D: row tiles
    (configs.heat3d_op, (6, 14, 124), 'zeros', MarchTuning(exchange=True, ry=2, ty=6), True, 4e-7),     # fused pair, rows exchanged
    (configs.stencil27_op, (5, 9, 60), None, MarchTuning(exchange=False, ry=2, ty=4, sx=2), True, 1e-14),  # fused pair, recomputed
    (configs.heat3d_op, (6, 40, 132), 'zeros', None, False, 3e-7),       # the shipped C3 geometry: 16+1 warps
    (configs.heat3d_op, (6, 50, 124), 'zeros', None, True, 4e-7),        # the shipped fused-pair geometry: 11+1 warps
    (configs.stencil27_op, (5, 25, 132), 'zeros', None, False, 1e-14),   # the shipped C4 geometry: 7+1 warps
])
def test_full_pipeline_replay(make, shape, bh, tuning, chain, tol):
    """csrc/kernels/psad_march.cuh itself — item loop, producer lane, slot / parity bookkeeping, expect_tx / complete_tx,
    slot release — with emulated mbarriers and TMA (tests/cpu_shim_full): several work items per CTA so that the ring
    wraps and the barrier phases flip across item boundaries."""
    op = make(shape=shape, boundary_handling=bh)
    ir = op.forward_ast_gpu
    ek = emit_march_chain(ir, tuning) if chain else emit_march(ir, tuning, masked=True)
    arrays, named = _fields(ek, ir, shape, seed=12)
    ctas, waits, loads = emu.run(ek, arrays, full=True, sm_count=2)
    fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
    ref = named[fin].copy()
    for _ in range(2 if chain else 1):
        ref = evaluate(op.forward_assignments, {fin: ref}, boundary_handling=bh)[fout].astype(ref.dtype)
    assert not np.isnan(named[fout]).any()
    np.testing.assert_allclose(named[fout], ref, rtol=0, atol=tol)
    # every staged plane was requested exactly once: items x planes per item (3-D: chunk + warm-up planes)
    assert ctas == 2 and loads > 2 * ek.geometry['STAGES'] and waits > loads


@pytest.mark.parametrize('case', ['z-only', 'yx-only', 'radius-2-x', 'pointwise'])
def test_fused_steps_degenerate_halos_replay(case):
    """Stencils without a z, y or x halo (one window phase, no rows to exchange, no columns to overlap) and a radius-2
    stencil (two radii exactly fill a strip) through the fused-pair emitter."""
    import pystencils_autodiff_b200 as ps
    shape = (5, 9, 60)
    u, out = ps.fields('u, out: float32[5,9,60]')
    rhs = {'z-only': 0.5 * u[0, 0, 0] + 0.25 * u[1, 0, 0] + 0.125 * u[-1, 0, 0],
           'yx-only': 0.6 * u[0, 0, 0] + 0.1 * (u[0, 1, 0] + u[0, -1, 0] + u[0, 0, 1] + u[0, 0, -1]),
           'radius-2-x': 0.5 * u[0, 0, 0] + 0.25 * u[0, 0, 2] + 0.25 * u[0, 0, -2],
           'pointwise': 0.5 * u[0, 0, 0] * u[0, 0, 0] + 0.1}[case]
    for bh in ('zeros', None):
        op = ps.AutoDiffOp(ps.AssignmentCollection([ps.Assignment(out.center, rhs)]), op_name='deg', boundary_handling=bh)
        ir = op.forward_ast_gpu
        ek = emit_march_chain(ir)
        assert ek.geometry['exchange'] == (case == 'never')       # no y halo or no z coupling: nothing to exchange
        arrays, named = _fields(ek, ir, shape, seed=6)
        emu.run(ek, arrays, full=(bh is None))
        ref = _twice(op.forward_assignments, 'u', 'out', named['u'].copy(), bh)
        np.testing.assert_allclose(named['out'], ref, rtol=1e-6, atol=1e-6)


def test_fused_steps_two_dimensional_lifted_replay():
    """2-D 'zeros' stencils reach the fused-pair emitter as 3-D fields of one plane (ir.lift_to_3d)."""
    from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
    shape = (45, 124)
    op = configs.diffusion2d_op(shape=shape)
    for ir, assigns in ((op.forward_ast_gpu, op.forward_assignments), (op.backward_ast_gpu, op.backward_assignments)):
        k = CompiledKernel(ir)
        assert k.fused_steps_reason() is None
        ek = k.emitted('march_x2')
        assert ek.plan['ndim'] == 3 and ek.plan['fused_steps'] == 2
        fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
        u = emu.aligned_empty((1,) + shape, np.float32)
        u[...] = np.random.default_rng(3).standard_normal((1,) + shape)
        out = emu.aligned_empty((1,) + shape, np.float32, np.nan)
        arrays = [out if f.name == fout else u for f in ek.fields]
        emu.run(ek, arrays, full=True)
        ref = _twice(assigns, fin, fout, u[0].copy(), 'zeros')
        np.testing.assert_allclose(out[0], ref, rtol=0, atol=4e-7)
    # interior iteration (boundary None) would also strip the new dimension: not offered
    assert CompiledKernel(configs.diffusion2d_op(shape=shape, boundary_handling=None).forward_ast_gpu).fused_steps_reason()


@pytest.mark.timeout(600)
@pytest.mark.parametrize('make, bh, world, tuning, full, tol', [
    (configs.heat3d_op, 'zeros', 2, None, False, 5e-7),                          # shipped fused geometry, rows exchanged
    (configs.heat3d_op, None, 3, MarchTuning(exchange=False), False, 5e-7),      # rows recomputed, global interior clipped
    (configs.stencil27_op, 'zeros', 2, MarchTuning(exchange=False, ry=2, ty=4, sx=2), True, 1e-14),   # real psad_march.cuh
    (configs.heat3d_op, None, 2, MarchTuning(exchange=True, ry=2, ty=6), True, 5e-7),                  # real psad_march.cuh
])
def test_slab_fused_steps_ranges_replay(make, bh, world, tuning, full, tol):
    """Two fused steps on slabs: every rank's interior / boundary launches of the fused-pair kernel over its slab with
    2 x halo ghost planes (datahandling.slab_ranges(..., steps=2)) reproduce the unsharded fused launch bit for bit —
    the iteration range bounds the intermediate field on the ghost planes, the write range the stored planes."""
    from pystencils_autodiff_b200.datahandling import slab_ranges
    n, g, G = 5, 1, 2
    shape = (n * world, 14 if full else 50, 68 if full else 132)
    op = make(shape=shape, boundary_handling=bh)
    ir = op.forward_ast_gpu
    dt = ir.input_fields[0].dtype.numpy_dtype
    rng = np.random.default_rng(11)
    u = emu.aligned_empty(shape, dt)
    u[...] = rng.standard_normal(shape)
    whole = emu.aligned_empty(shape, dt, np.nan)
    emu.run(emit_march_chain(ir, tuning), [whole, u])
    ref = _twice(op.forward_assignments, 'u', 'out', u.copy(), bh)
    np.testing.assert_allclose(whole, ref, rtol=0, atol=tol)
    for rank in range(world):
        start = rank * n
        local_u = emu.aligned_empty((n + 2 * G,) + shape[1:], dt, 0.0)
        lo, hi = max(0, start - G), min(shape[0], start + n + G)
        local_u[lo - (start - G):hi - (start - G)] = u[lo:hi]        # owned planes + received ghost planes
        local_out = emu.aligned_empty(local_u.shape, dt, np.nan)
        local_kernel = emit_march_chain(make(shape=local_u.shape, boundary_handling=bh).forward_ast_gpu, tuning)
        parts = slab_ranges(shape, start, n, G, rank > 0, rank < world - 1, 'zeros' if bh == 'zeros' else 'none',
                            ir.ghost_layers, 3, steps=2, halo=g)
        written = np.zeros(n + 2 * G, dtype=int)
        for part in parts:
            if part is None:
                continue
            written[part['write_lo'][0]:part['write_hi'][0]] += 1
            emu.run(local_kernel, [local_out, local_u], launch_range=part, full=full)
        assert list(written) == [0] * G + [1] * n + [0] * G
        assert np.array_equal(local_out[G:G + n], whole[start:start + n]), rank
        assert np.isnan(local_out[:G]).all() and np.isnan(local_out[G + n:]).all()      # ghost planes are not written


def test_slab_ranges_fused_steps_preconditions():
    from pystencils_autodiff_b200.datahandling import slab_ranges
    with pytest.raises(ValueError, match='ghost planes'):
        slab_ranges((12, 8, 8), 6, 6, 1, True, False, 'zeros', 0, 3, steps=2, halo=1)
    with pytest.raises(ValueError, match='too thin'):
        slab_ranges((12, 8, 8), 4, 3, 2, True, True, 'zeros', 0, 3, steps=2, halo=1)
    # a single rank needs no ghost planes at all
    interior, lo, hi = slab_ranges((12, 8, 8), 0, 12, 0, False, False, 'zeros', 0, 3, steps=2, halo=1)
    assert lo is None and hi is None and interior['write_lo'] == [0, 0, 0] and interior['iter_hi'] == [12, 8, 8]


def _golden_march_names():
    from golden_util import golden_names
    return [n for n in golden_names() if n.endswith('_aligned') or n.startswith('random_')]


@pytest.mark.parametrize('name', _golden_march_names())
def test_march_kernels_against_reference_golden_vectors(name):
    """The emitted march kernels (CPU replay) against the committed golden vectors — outputs and gradients of the
    REFERENCE's own forward / backward assignments (tests/golden/make_reference_golden.py) on seeded float64 inputs."""
    from golden_util import build_op, golden_arrays
    from pystencils_autodiff_b200.emit import march_ineligible_reason
    ran = 0
    for mode in (None, 'zeros'):
        op = build_op(name, mode)
        ins, outs, grads = golden_arrays(name, mode)
        for ir, gold in ((op.forward_ast_gpu, outs), (op.backward_ast_gpu, grads)):
            if march_ineligible_reason(ir):
                continue
            try:
                ek = emit_march(ir, None, masked=True)
            except ValueError:
                continue
            arrays, named = [], {}
            for f in ek.fields:
                shape = next(iter(ins.values())).shape
                a = emu.aligned_empty(shape, f.dtype.numpy_dtype, np.nan)
                if f in ir.input_fields:
                    a[...] = ins[f.name]
                arrays.append(a)
                named[f.name] = a
            emu.run(ek, arrays)
            for f in ir.output_fields:
                scale = max(1.0, np.abs(gold[f.name]).max())
                assert np.abs(named[f.name] - gold[f.name]).max() <= 1e-12 * scale, (name, mode, f.name)
                ran += 1
    if name.endswith('_aligned'):
        assert ran >= 4            # forward + adjoint, both boundary modes


def test_exact_adjoint_mode_tv_kernel_replay():
    """``adjoint_mode='exact'`` (shifted coefficients: the true transpose for non-linear stencils) goes through the same
    march emitter: the TV-gradient adjoint kernel of that mode against the oracle on its own assignments."""
    shape = (2, 33, 132)
    op = configs.tv_gradient_op(shape=shape, adjoint_mode='exact')
    ir = op.backward_ast_gpu
    ek = emit_march(ir, None, masked=True)
    rng = np.random.default_rng(0)
    arrays, named = [], {}
    for f in ek.fields:
        a = emu.aligned_empty(shape, f.dtype.numpy_dtype)
        a[...] = rng.random(shape) if f in ir.input_fields else np.nan
        arrays.append(a)
        named[f.name] = a
    emu.run(ek, arrays)
    ref = evaluate(op.backward_assignments, {f.name: named[f.name].copy() for f in ir.input_fields}, boundary_handling='zeros')
    for f in ir.output_fields:
        assert np.abs(named[f.name] - ref[f.name]).max() <= 2e-6 * max(1.0, np.abs(ref[f.name]).max())
