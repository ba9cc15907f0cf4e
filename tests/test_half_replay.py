"""float16 fields (fp16 storage, fp32 arithmetic) without a GPU: NVRTC compiles of the march and generic kernels, the
real march template and the generic kernels replayed on the CPU (tests/march_emulator.py, host stand-ins in
tests/cpu_shim*/psad_half.cuh), launch planning with 2-byte fields, a two-rank slab time loop, and the cases this
release declines (fused pairs, peer halos).

Accuracy policy (DESIGN §6): max |got - ref| / max |ref| <= 5e-4, the reference being the fp64 oracle evaluated on the
fp16 inputs converted exactly to fp64 — one fp16 rounding of the result (at most 2^-11 of the largest value) plus the fp32
allowance.  Time loops compare against a step-by-step oracle that rounds to fp16 after every step (STEPS_TOL)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import march_emulator as emu
from oracle.evaluate import evaluate
from pystencils_autodiff_b200 import configs, runtime
from pystencils_autodiff_b200.emit import MarchTuning, emit_generic, emit_march, march_ineligible_reason

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HALF_TOL = 5e-4
# time loops: an fp32 and an fp64 result can round to neighbouring halves in one step, and the step after carries that
# difference on — against the oracle rounded after every step, one fp16 spacing (2^-10 ~ 9.8e-4) of the largest value
STEPS_TOL = 1e-3
F16 = np.float16


def _rel_err(got, ref):
    return float(np.abs(got.astype(np.float64) - ref).max() / max(1e-30, np.abs(ref).max()))


def _ops(make, shape, bh):
    """The float16 op and its float64 twin (same stencil, same field names): the twin's assignments are the oracle."""
    return make(shape=shape, dtype='float16', boundary_handling=bh), make(shape=shape, dtype='float64', boundary_handling=bh)


def _inputs(ek, ir, shape, seed):
    rng = np.random.default_rng(seed)
    arrays, named = [], {}
    for f in ek.fields:
        a = emu.aligned_empty(shape, f.dtype.numpy_dtype)
        a[...] = rng.uniform(0.5, 1.5, size=shape) if f in ir.input_fields else np.nan
        arrays.append(a)
        named[f.name] = a
    return arrays, named


def _rounded_steps(op64, u, steps, bh):
    """Step-by-step oracle of a time loop: fp64 steps, each result rounded to fp16 (as the kernels store it)."""
    ref = u.astype(np.float64)
    for _ in range(steps):
        ref = evaluate(op64.forward_assignments, {'u': ref}, bh)['out'].astype(F16).astype(np.float64)
    return ref


def _oracle(op64, which, named, ir, bh):
    assigns = op64.forward_assignments if which == 'forward' else op64.backward_assignments
    return evaluate(assigns, {f.name: named[f.name].astype(np.float64) for f in ir.input_fields}, boundary_handling=bh)


# ---- NVRTC for sm_100a, no GPU -------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['c2', 'c3', 'c4', 'c5'])
def test_half_kernels_compile_without_spills(name):
    from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
    shape = {'c2': (64, 128), 'c3': (8, 16, 128), 'c4': (8, 16, 128), 'c5': (2, 16, 128)}[name]
    for bh in (None, 'zeros'):
        op = configs.make_config(name, shape=shape, dtype='float16', boundary_handling=bh)
        for ir in (op.forward_ast_gpu, op.backward_ast_gpu):
            k = CompiledKernel(ir)
            assert k._march_reason is None and set(k._emitted) == {'march', 'march_nomask', 'generic'}
            for variant, ek in k._emitted.items():
                assert '#include "psad_half.cuh"' in ek.source and 'cuda_fp16' not in ek.source
                key = ek.cache_key + '_spills'        # a key of its own: a cache hit would return no ptxas log
                _, log = runtime.compile_source(ek.source, key, list(ek.options) + ['--ptxas-options=-v'])
                os.remove(runtime.cubin_path(key))
                spills = [ln for ln in log.splitlines() if ln.startswith('ptxas') and 'spill' in ln]
                assert spills and all(' 0 bytes spill stores, 0 bytes spill loads' in ln for ln in spills), (variant, spills)


def test_half_march_geometry_and_cache_key():
    op = configs.heat3d_op(shape=(8, 16, 128), dtype='float16')
    ek = emit_march(op.forward_ast_gpu)
    # 4 cells per lane (one 8-byte vector), pads in 16-byte units: the box is 128 + 2 x 8 halves wide
    assert ek.geometry['SX'] == 4 and ek.geometry['TX'] == 128
    assert [f['box'] for f in ek.plan['fields'] if f['tma']] == [(144, 34, 1)]
    assert all(f['elem_size'] == 2 for f in ek.plan['fields'])
    assert 'psad_lds_h4' in ek.source and 'psad_stg_h4' in ek.source
    # the half helpers are part of the key of the kernels that include them, and of no other kernel's key
    import hashlib
    from pystencils_autodiff_b200 import emit as emit_mod
    op32 = configs.heat3d_op(shape=(8, 16, 128))
    ek32 = emit_march(op32.forward_ast_gpu)
    h = hashlib.md5()
    h.update(emit_mod.EMITTER_VERSION.encode())
    h.update(ek32.source.encode())
    h.update(' '.join(ek32.options).encode())
    for fn in sorted(os.listdir(emit_mod.KERNEL_DIR)):
        if fn != 'psad_half.cuh':
            with open(os.path.join(emit_mod.KERNEL_DIR, fn), 'rb') as fh:
                h.update(fh.read())
    assert ek32.cache_key.endswith(h.hexdigest())
    assert not ek.cache_key.endswith(h.hexdigest())


def test_half_eligibility():
    import pystencils_autodiff_b200 as ps
    u = ps.fields('u: float16[16,128]')
    o = ps.fields('o: float32[16,128]')
    op = ps.AutoDiffOp([ps.Assignment(o.center, u[1, 0] + u[-1, 0] - 2 * u[0, 0])], op_name='mix', boundary_handling='zeros')
    assert march_ineligible_reason(op.forward_ast_gpu) == 'float16 fields mixed with wider fields'
    assert op.forward_ast_gpu.compute_dtype == np.float32
    op16 = configs.heat3d_op(shape=(4, 8, 128), dtype='float16')
    assert march_ineligible_reason(op16.forward_ast_gpu) is None
    assert op16.forward_ast_gpu.compute_dtype == np.float32
    assert op16.forward_ast_gpu.bytes_per_cell() == 4


# ---- the real march template on the CPU ------------------------------------------------------------------------------------
@pytest.mark.timeout(600)
@pytest.mark.parametrize('make, shape, bh, which, tuning', [
    (configs.heat3d_op, (9, 13, 136), 'zeros', 'forward', MarchTuning(ry=2, ty=6)),
    (configs.heat3d_op, (7, 11, 264), None, 'backward', MarchTuning(ry=1, ty=3, lookahead=1)),
    (configs.heat3d_op, (5, 40, 136), 'zeros', 'backward', None),              # the shipped geometry: 16+1 warps
    (configs.stencil27_op, (6, 9, 72), 'zeros', 'forward', MarchTuning(ry=3, ty=6)),
    (configs.stencil27_op, (5, 10, 136), None, 'backward', MarchTuning(ry=2, ty=4)),
    (configs.diffusion2d_op, (23, 136), 'zeros', 'forward', MarchTuning(ry=1, ty=4)),
    (configs.diffusion2d_op, (21, 264), None, 'backward', MarchTuning(ry=1, ty=4)),
    (configs.tv_gradient_op, (3, 11, 136), 'zeros', 'forward', MarchTuning(ry=2, ty=4)),
    (configs.tv_gradient_op, (3, 9, 136), None, 'backward', MarchTuning(ry=1, ty=3)),
])
def test_half_full_pipeline_replay(make, shape, bh, which, tuning):
    """csrc/kernels/psad_march.cuh with fp16 boxes: TMA staging of 2-byte elements, 8-byte shared loads converted into the
    fp32 register window, shuffled x-halos, packed fp16 stores; masked and mask-free instances, ragged y / z extents."""
    op16, op64 = _ops(make, shape, bh)
    ir = op16.forward_ast_gpu if which == 'forward' else op16.backward_ast_gpu
    for masked in (True, False):
        if not masked and bh is None:
            continue          # 'none' boundary: the written cells reach beyond the iterated ones, only the masked instance
        ek = emit_march(ir, tuning, masked=masked)
        arrays, named = _inputs(ek, ir, shape, seed=3)
        ctas, waits, loads = emu.run(ek, arrays, full=True, sm_count=2)
        assert ctas == 2 and loads > 0
        ref = _oracle(op64, which, named, ir, bh)
        for f in ir.output_fields:
            got = named[f.name]
            assert got.dtype == F16 and not np.isnan(got).any()
            assert _rel_err(got, ref[f.name]) <= HALF_TOL, (f.name, masked, _rel_err(got, ref[f.name]))


@pytest.mark.parametrize('which', ['forward', 'backward'])
def test_half_march_matches_generic(which):
    """The march kernel (plane sums, shared partial sums) and the generic kernel (one FMA chain per cell) evaluate the
    27-point sum in different orders: their fp16 results differ by at most one rounding step."""
    shape = (6, 18, 136)
    op16, _ = _ops(configs.stencil27_op, shape, 'zeros')
    ir = op16.forward_ast_gpu if which == 'forward' else op16.backward_ast_gpu
    ek = emit_march(ir, MarchTuning(ry=2, ty=6), masked=False)
    arrays, named = _inputs(ek, ir, shape, seed=8)
    emu.run(ek, arrays)
    gen = emit_generic(ir)
    arrays_g = [a.copy() for a in arrays]
    for f, a in zip(gen.fields, arrays_g):
        if f in ir.output_fields:
            a[...] = np.nan
    emu.run_generic(gen, arrays_g)
    for f, a, b in zip(ek.fields, arrays, arrays_g):
        if f in ir.output_fields:
            assert _rel_err(a, b.astype(np.float64)) <= 2.0 ** -10
            assert np.mean(a != b) < 0.05
        else:
            assert np.array_equal(a, b)


# ---- generic kernels -----------------------------------------------------------------------------------------------------
def test_half_generic_strided_views_and_launch_range():
    import pystencils_autodiff_b200 as ps
    u, out = ps.fields('u, out: float16[9,14]')
    u64, out64 = ps.fields('u, out: float64[9,14]')
    ex = lambda u_, o_: [ps.Assignment(o_.center, 0.5 * u_[0, 0] + 0.25 * u_[1, -2] - u_[-1, 1] * u_[0, 1])]   # noqa: E731
    op = ps.AutoDiffOp(ex(u, out), op_name='strided16', boundary_handling='zeros')
    op64 = ps.AutoDiffOp(ex(u64, out64), op_name='strided64', boundary_handling='zeros')
    ek = emit_generic(op.forward_ast_gpu)
    rng = np.random.default_rng(1)
    ut = np.asfortranarray(rng.uniform(-1, 1, (9, 14)).astype(F16))    # x is NOT the contiguous axis
    big = np.full((9, 21), np.nan, dtype=F16)
    ot = big[:, 3:17]                                                  # row pitch 21 halves: unaligned rows
    emu.run_generic(ek, [ot, ut])
    ref = evaluate(op64.forward_assignments, {'u': np.ascontiguousarray(ut).astype(np.float64)}, 'zeros')['out']
    assert _rel_err(ot, ref) <= HALF_TOL
    assert np.isnan(big[:, :3]).all() and np.isnan(big[:, 17:]).all()
    ot2 = np.full((9, 14), np.nan, dtype=F16)
    emu.run_generic(ek, [ot2, ut], launch_range=dict(iter_lo=[3, 2], iter_hi=[6, 14], write_lo=[2, 0], write_hi=[7, 14]))
    assert np.isnan(ot2[:2]).all() and np.isnan(ot2[7:]).all()
    assert np.all(ot2[2] == 0) and np.all(ot2[6] == 0) and np.all(ot2[3:6, :2] == 0)
    assert np.abs(ot2[3:6, 2:].astype(np.float64) - ref[3:6, 2:]).max() <= HALF_TOL * np.abs(ref).max()


def test_half_generic_index_dimension_and_mixed_precision():
    import pystencils_autodiff_b200 as ps
    disc = ps.fd.Discretization2ndOrder(dx=1)

    def curl(dt_u, dt_c):
        u = ps.Field.create_fixed_size('u', (8, 12), index_dimensions=0, dtype=dt_u)
        c = ps.Field.create_fixed_size('c', (8, 12, 2), index_dimensions=1, dtype=dt_c)
        return ps.AutoDiffOp(ps.AssignmentCollection([ps.Assignment(c.center(0), disc(ps.fd.Diff(u, 0))),
                                                      ps.Assignment(c.center(1), disc(ps.fd.Diff(u, 1)))], []),
                             op_name='curl', boundary_handling='zeros')
    U = np.random.default_rng(3).uniform(-1, 1, (8, 12)).astype(F16)
    ref = evaluate(curl(np.float64, np.float64).forward_assignments, {'u': U.astype(np.float64)}, 'zeros')['c']
    # all float16 (index dimension, array-of-structures layout), and float16 input with a float32 output
    for dt_c in (F16, np.float32):
        op = curl(F16, dt_c)
        ir = op.forward_ast_gpu
        assert ir.compute_dtype == np.float32
        ek = emit_generic(ir)
        C = np.full((8, 12, 2), np.nan, dtype=dt_c)
        emu.run_generic(ek, [C if f.name == 'c' else U for f in ek.fields])
        assert _rel_err(C, ref) <= (HALF_TOL if dt_c == F16 else 2e-6), dt_c
    # fp32 input, fp16 output, and the adjoint of the mixed kernel (diffu float16 from a float32 gradient)
    op = curl(F16, np.float32)
    ir = op.backward_ast_gpu
    assert march_ineligible_reason(ir) is not None
    G = np.random.default_rng(4).uniform(-1, 1, (8, 12, 2)).astype(np.float32)
    ek = emit_generic(ir)
    D = np.full((8, 12), np.nan, dtype=F16)
    emu.run_generic(ek, [D if f.name == 'diffu' else G for f in ek.fields])
    refd = evaluate(curl(np.float64, np.float64).backward_assignments, {'diffc': G.astype(np.float64)}, 'zeros')['diffu']
    assert _rel_err(D, refd) <= HALF_TOL


def test_half_data_type_double():
    """``data_type='double'``: fp64 arithmetic on fp16 storage, one rounding from fp64 per cell."""
    from pystencils_autodiff_b200.ir import lower_assignments
    shape = (5, 12, 136)
    op16 = configs.heat3d_op(shape=shape, dtype='float16', boundary_handling='zeros')
    ir = lower_assignments(op16.forward_assignments, 'zeros', 'heat_d', data_type='double')
    assert ir.compute_dtype == np.float64
    _, op64 = _ops(configs.heat3d_op, shape, 'zeros')
    ek = emit_march(ir, MarchTuning(ry=2, ty=6), masked=False)
    assert 'typedef double CT;' in ek.source
    arrays, named = _inputs(ek, ir, shape, seed=5)
    emu.run(ek, arrays, full=True, sm_count=2)
    ref = _oracle(op64, 'forward', named, ir, 'zeros')['out']
    # one rounding from fp64 per cell.  Not bitwise the oracle's own fp16 store: with fp16 inputs and alpha = 0.1 many
    # exact results are ties (k + 1/2 fp16 spacings), and two fp64 sums in different orders round those either way
    assert _rel_err(named['out'], ref) <= HALF_TOL


# ---- launch planning ---------------------------------------------------------------------------------------------------
def test_plan_launch_with_two_byte_fields():
    import ctypes
    op = configs.heat3d_op(shape=(4, 8, 136), dtype='float16')
    ek = emit_march(op.forward_ast_gpu)
    L = runtime.lib()
    plan = runtime.make_plan(ek.plan)

    def plan_for(shape, row_pitch):
        fa = (runtime.FieldArg * 2)()
        buf = emu.aligned_empty((shape[0] * shape[1] * row_pitch + 64,), F16)
        for i in range(2):
            fa[i].ptr = buf.ctypes.data
            fa[i].shape[:] = list(shape)
            fa[i].stride[:] = [shape[1] * row_pitch, row_pitch, 1, 0]
        args = ctypes.create_string_buffer(4096)
        grid = (ctypes.c_uint * 3)()
        sc = (ctypes.c_double * 1)()
        return L.psad_plan_launch(ctypes.byref(plan), 4, 1, fa, 2, sc, 0, None, args, emu._args_size(), grid), grid
    rc, grid = plan_for((4, 8, 136), 136)
    assert rc == 0 and grid[0] > 0
    rc, _ = plan_for((4, 8, 132), 132)        # 264-byte rows: not a multiple of 16 bytes
    assert rc != 0 and '16 bytes' in runtime.lib().psad_last_error().decode()


# ---- declined in this release ------------------------------------------------------------------------------------------
def test_half_fused_pairs_declined():
    from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
    from pystencils_autodiff_b200.datahandling import SlabDataHandling
    from replay_kernels import ReplayKernel
    shape = (4, 16, 136)
    op16, op64 = _ops(configs.heat3d_op, shape, 'zeros')
    k = ReplayKernel(op16.forward_ast_gpu)
    assert k.fused_steps_reason() == 'float16 fields: fused pairs not implemented'
    with pytest.raises(ValueError, match='float16 fields: fused pairs not implemented'):
        k.emitted('march_x2')
    u0 = np.random.default_rng(2).uniform(-1, 1, shape).astype(F16)
    src = torch.from_numpy(u0)
    with pytest.raises(ValueError, match='float16'):
        k.run_steps(src, 4, fuse=True)
    ReplayKernel.launches.clear()
    out = k.run_steps(src, 3)                                   # default: single steps
    assert ReplayKernel.launches == ['psad_heat3d_forward_gpu_march_nomask'] * 3
    assert _rel_err(out.numpy(), _rounded_steps(op64, u0, 3, 'zeros')) <= STEPS_TOL
    dh = SlabDataHandling(shape, 0, 1, 0, device='cpu', backend='torch')
    dh.add_arrays('u, out', dtype=F16)
    for fuse in (None, True):
        tl = dh.create_timeloop(fuse_steps=fuse)
        tl.add_call(CompiledKernel(op16.forward_ast_gpu), {})
        tl.swap('u', 'out')
        if fuse:
            with pytest.raises(ValueError, match='float16'):
                tl.fused_pair()
        else:
            assert tl.fused_pair() is None


class _StubPeer:
    """Stands in for the CUDA IPC machinery: records what would be registered."""

    def __init__(self, dh):
        self.registered = []

    def register(self, t):
        self.registered.append(t)

    def close(self):
        pass


def _slab_worker(rank, world, port, steps, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from pystencils_autodiff_b200 import datahandling
        from pystencils_autodiff_b200.datahandling import SlabDataHandling
        from replay_kernels import ReplayKernel
        gshape = (5 * world, 14, 136)
        glob_u = np.random.default_rng(7).uniform(-1, 1, gshape).astype(F16)
        res = {}
        for bh in ('zeros', None):
            dh = SlabDataHandling(gshape, rank, world, 1, device='cpu', backend='torch')
            dh.add_arrays('u, out', dtype=F16)
            op_l = configs.heat3d_op(shape=dh.dec.local_shape, dtype='float16', boundary_handling=bh)
            kernel = ReplayKernel(op_l.forward_ast_gpu)
            sl = slice(dh.dec.start, dh.dec.start + dh.dec.n_local)
            dh.owned('u').copy_(torch.from_numpy(glob_u[sl]))
            ReplayKernel.launches.clear()
            tl = dh.create_timeloop()
            tl.add_call(kernel, {'halo_fields': ['u']})
            tl.swap('u', 'out')
            tl.run(steps)
            assert not tl.fused_last_run
            parts = 1 + int(rank > 0) + int(rank < world - 1)
            assert len(ReplayKernel.launches) == parts * steps and all('march' in n for n in ReplayKernel.launches)
            res[bh] = dh.gather_array('u')
        # peer halos: refused outright for float16 arrays
        orig = datahandling._PeerHalo
        datahandling._PeerHalo = _StubPeer
        try:
            dh = SlabDataHandling(gshape, rank, world, 1, device='cpu', backend='torch', peer_halo=True)
            assert dh.peer is not None
            dh.add_array('a32', dtype=np.float32)
            try:
                dh.add_array('a16', dtype=F16)
                peer_error = None
            except ValueError as e:
                peer_error = str(e)
            assert len(dh.peer.registered) == 1
        finally:
            datahandling._PeerHalo = orig
        q.put((rank, res, peer_error))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_half_slab_time_loop_two_ranks():
    """Two gloo ranks, ghost planes exchanged as fp16, single-step TimeLoop on the replayed march kernels against the
    step-by-step oracle rounded to fp16 after every step; ``peer_halo=True`` refuses float16 arrays."""
    world, steps = 2, 3
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29150                     # outside the ranges the other multi-process tests draw from
    procs = [ctx.Process(target=_slab_worker, args=(r, world, port, steps, q)) for r in range(world)]
    for p in procs:
        p.start()
    import test_slab_gloo
    results = test_slab_gloo._collect(procs, q, world)
    gshape = (5 * world, 14, 136)
    glob_u = np.random.default_rng(7).uniform(-1, 1, gshape).astype(F16)
    for bh in ('zeros', None):
        op64 = configs.heat3d_op(shape=gshape, dtype='float64', boundary_handling=bh)
        ref = _rounded_steps(op64, glob_u, steps, bh)
        for rank, res, peer_error in results:
            assert res[bh].dtype == F16
            assert _rel_err(res[bh], ref) <= STEPS_TOL, (bh, rank)
            assert peer_error is not None and 'float16' in peer_error
