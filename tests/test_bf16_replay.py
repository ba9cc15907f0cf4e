"""bfloat16 fields (bf16 storage, fp32 arithmetic) without a GPU: dtype plumbing, NVRTC compiles of the march and generic
kernels, the march template and the generic kernels replayed on the CPU (tests/march_emulator.py), the step decisions
this release declines (fused pairs, peer halos) and a two-rank slab time loop.

The replays compile against copies of the tests/cpu_shim*/ directories whose psad_half.cuh also defines host stand-ins for
the bfloat16 helpers (``BF16_HOST`` below, on g++'s ``__bf16``), see ``use_bf16_shims``.

numpy has no bfloat16: the replays hold bf16 cells as their raw 16-bit words (uint16 arrays), and bf16 tensors reach the
replayed kernels as int16 views of the same storage.

Accuracy policy (DESIGN §6): max |got - ref| / max |ref| <= 4e-3, the reference being the fp64 oracle evaluated on the
bf16 inputs converted exactly to fp64: one bf16 rounding of the result (at most 2^-8 of the largest value) plus the fp32
allowance.  Time loops compare against a step-by-step oracle that rounds to bf16 after every step, at one bf16 spacing
(2^-7).  torch rounds float64 -> bfloat16 through float32 (two roundings), so no comparison here is bit for bit against a
result rounded by torch."""
import os
import shutil
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
from pystencils_autodiff_b200.field import BFLOAT16
from replay_kernels import ReplayKernel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF16_TOL = 4e-3
STEPS_TOL = 8e-3
FUSE_REASON = 'bfloat16 fields: fused pairs not implemented'

# Host stand-ins for the bfloat16 part of csrc/kernels/psad_half.cuh.  g++'s __bf16 rounds to nearest even like cvt.rn,
# and double -> __bf16 rounds once like cvt.rn.bf16.f64, so the replay rounds every stored cell as the device does.
BF16_HOST = r"""
struct psad_bf16 {
  unsigned short bits;
  psad_bf16() = default;
  psad_bf16(float f) { const __bf16 b = (__bf16)f; std::memcpy(&bits, &b, 2); }
  psad_bf16(double d) { const __bf16 b = (__bf16)d; std::memcpy(&bits, &b, 2); }
  operator float() const { __bf16 b; std::memcpy(&b, &bits, 2); return (float)b; }
};

static inline void psad_lds_h4(const psad_bf16* p, float* e) {
  for (int i = 0; i < 4; ++i) e[i] = (float)p[i];
}
static inline void psad_stg_h4(psad_bf16* p, const float* e) {
  for (int i = 0; i < 4; ++i) p[i] = psad_bf16(e[i]);
}
static inline void psad_stg_h4(psad_bf16* p, const double* e) {
  for (int i = 0; i < 4; ++i) p[i] = psad_bf16(e[i]);
}
"""
_SHIM_DIRS = {attr: getattr(emu, attr) for attr in ('_SHIM', '_SHIM_FULL', '_SHIM_GENERIC')}


def bf16_shim_dirs(root):
    """Copies of the tests/cpu_shim*/ directories under ``root`` whose psad_half.cuh also holds ``BF16_HOST``;
    returns ``{march_emulator attribute: directory}``."""
    dirs = {}
    for attr, src in _SHIM_DIRS.items():
        dst = os.path.join(str(root), os.path.basename(src))
        if not os.path.isdir(dst):
            tmp = dst + '.tmp%d' % os.getpid()
            shutil.copytree(src, tmp)
            path = os.path.join(tmp, 'psad_half.cuh')
            with open(path) as fh:
                text = fh.read()
            cut = text.rindex('#endif')
            with open(path, 'w') as fh:
                fh.write(text[:cut] + BF16_HOST + '\n' + text[cut:])
            os.replace(tmp, dst)
        dirs[attr] = dst
    return dirs


def use_bf16_shims(root, monkeypatch=None):
    """Points the CPU replays (tests/march_emulator.py) at the shim copies with the bfloat16 stand-ins."""
    for attr, d in bf16_shim_dirs(root).items():
        if monkeypatch is None:
            setattr(emu, attr, d)
        else:
            monkeypatch.setattr(emu, attr, d)


@pytest.fixture(scope='module', autouse=True)
def _bf16_shims(tmp_path_factory):
    root = tmp_path_factory.mktemp('bf16_shims')
    with pytest.MonkeyPatch.context() as mp_:
        use_bf16_shims(root, mp_)
        yield root


def to_words(x):
    """float values -> bf16 words (uint16), rounded to nearest even from float32."""
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16)
    return t.view(torch.int16).numpy().view(np.uint16)


def from_words(w):
    """bf16 words -> float64 (exact)."""
    return (np.asarray(w).astype(np.uint32) << 16).view(np.float32).astype(np.float64)


def round_bf16(x):
    """float64 -> nearest bf16 value, as float64 (through float32, as torch does)."""
    return torch.from_numpy(np.asarray(x, dtype=np.float64)).to(torch.bfloat16).double().numpy()


def _rel_err(got, ref):
    return float(np.abs(got - ref).max() / max(1e-300, np.abs(ref).max()))


class BF16Replay(ReplayKernel):
    """The replayed launch on bf16 tensors: numpy cannot hold bfloat16, so the kernel sees int16 views of the same
    storage (the emitted kernel reads and writes raw 16-bit words either way)."""

    def __call__(self, **kwargs):
        kwargs = {k: (v.detach().view(torch.int16) if isinstance(v, torch.Tensor) and v.dtype == torch.bfloat16 else v)
                  for k, v in kwargs.items()}
        return super().__call__(**kwargs)


def _ops(make, shape, bh):
    """The bfloat16 op and its float64 twin (same stencil, same field names): the twin's assignments are the oracle."""
    return make(shape=shape, dtype='bfloat16', boundary_handling=bh), make(shape=shape, dtype='float64', boundary_handling=bh)


def _inputs(ek, ir, shape, seed, scale=1.0):
    """Arrays in plan order: bf16 words for bf16 fields (inputs random, outputs NaN words), named float64 inputs."""
    rng = np.random.default_rng(seed)
    arrays, named = [], {}
    for f in ek.fields:
        bf = f.dtype.numpy_dtype == BFLOAT16
        a = emu.aligned_empty(shape, np.uint16 if bf else f.dtype.numpy_dtype)
        if f in ir.input_fields:
            v = rng.uniform(0.5, 1.5, size=shape) * scale
            a[...] = to_words(v) if bf else v
            named[f.name] = from_words(a) if bf else a.astype(np.float64)
        else:
            a[...] = 0x7fc1 if bf else np.nan
        arrays.append(a)
    return arrays, named


def _oracle(op64, which, named, bh):
    assigns = op64.forward_assignments if which == 'forward' else op64.backward_assignments
    return evaluate(assigns, named, boundary_handling=bh)


def _rounded_steps(op64, u, steps, bh):
    """Step-by-step oracle of a time loop: fp64 steps, each result rounded to bf16 (as the kernels store it)."""
    ref = np.asarray(u, dtype=np.float64)
    for _ in range(steps):
        ref = round_bf16(evaluate(op64.forward_assignments, {'u': ref}, bh)['out'])
    return ref


# ---- dtype plumbing ------------------------------------------------------------------------------------------------------
def test_bf16_dtype_plumbing():
    import pystencils_autodiff_b200 as ps
    from pystencils_autodiff_b200.backends._torch_native import numpy_dtype_to_torch
    from pystencils_autodiff_b200.datahandling import SlabDataHandling
    from pystencils_autodiff_b200.field_tensor_conversion import create_field_from_array_like, torch_tensor_from_field
    u, out = ps.fields('u, out: bfloat16[4,8]')
    assert u.dtype.numpy_dtype == BFLOAT16 and u.dtype.itemsize == 2 and str(u.dtype) == 'bfloat16'
    assert numpy_dtype_to_torch(BFLOAT16) is torch.bfloat16 and numpy_dtype_to_torch('bfloat16') is torch.bfloat16
    assert numpy_dtype_to_torch(np.float16) is torch.float16 and numpy_dtype_to_torch('float32') is torch.float32
    t = torch_tensor_from_field(out, cuda=False)
    assert t.dtype == torch.bfloat16 and t.shape == (4, 8)
    x = torch.zeros(6, 10, dtype=torch.bfloat16)[:, 1:9]
    fx = ps.fields(x=x)
    assert fx.dtype.numpy_dtype == BFLOAT16 and fx.shape == (6, 8) and fx.strides == (10, 1)
    assert create_field_from_array_like('y', x).dtype.numpy_dtype == BFLOAT16
    # the compute type: fp32 for bf16 fields alone or with fp16 / fp32 ones, fp64 with an fp64 field or data_type='double'
    lap = lambda a, o: [ps.Assignment(o.center, a[1, 0] + a[-1, 0] - 2 * a[0, 0])]    # noqa: E731
    for dt_o, expected in (('bfloat16', np.float32), ('float16', np.float32), ('float32', np.float32),
                           ('float64', np.float64)):
        o = ps.fields('o: %s[4,8]' % dt_o)
        assert ps.AutoDiffOp(lap(u, o), op_name='cd').forward_ast_gpu.compute_dtype == expected, dt_o
    assert ps.AutoDiffOp(lap(u, out), op_name='cdd', data_type='double').forward_ast_gpu.compute_dtype == np.float64
    op3 = configs.make_config('c3', shape=(4, 8, 128), dtype='bfloat16')
    assert op3.forward_ast_gpu.compute_dtype == np.float32 and op3.forward_ast_gpu.bytes_per_cell() == 4
    # slab data handling: bf16 arrays, add_array_like, float32 host copies
    dh = SlabDataHandling((4, 8), 0, 1, 1, device='cpu', backend='torch')
    dh.add_arrays('a, b', dtype='bfloat16')
    assert dh.gpu_arrays['a'].dtype == torch.bfloat16 and dh.fields['a'].dtype.numpy_dtype == BFLOAT16
    dh.add_array_like('c', 'a')
    assert dh.gpu_arrays['c'].dtype == torch.bfloat16
    dh.add_arrays('d: bfloat16[4,8]')
    assert dh.gpu_arrays['d'].dtype == torch.bfloat16
    dh.fill('a', 1e-9)
    g = dh.gather_array('a')
    assert g.dtype == np.float32 and g.shape == (4, 8) and np.all(g == torch.tensor(1e-9, dtype=torch.bfloat16).item())


def test_bf16_save_fields(tmp_path):
    from pystencils_autodiff_b200.datahandling import SlabDataHandling
    dh = SlabDataHandling((4, 8), 0, 1, 1, device='cpu', backend='torch')
    dh.add_arrays('a', dtype='bfloat16')
    dh.fill('a', 3e7)
    dh.save_fields(['a'], str(tmp_path / 'snap'))
    a = np.load(str(tmp_path / 'snap.rank0.npz'))['a']
    assert a.dtype == np.float32 and np.all(a == torch.tensor(3e7, dtype=torch.bfloat16).item())


# ---- NVRTC for sm_100a, no GPU -------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['c2', 'c3', 'c4', 'c5'])
def test_bf16_kernels_compile_without_spills(name):
    from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
    shape = {'c2': (64, 128), 'c3': (8, 16, 128), 'c4': (8, 16, 128), 'c5': (2, 16, 128)}[name]
    for bh in (None, 'zeros'):
        op = configs.make_config(name, shape=shape, dtype='bfloat16', boundary_handling=bh)
        for ir in (op.forward_ast_gpu, op.backward_ast_gpu):
            k = CompiledKernel(ir)
            assert k._march_reason is None and set(k._emitted) == {'march', 'march_nomask', 'generic'}
            for variant, ek in k._emitted.items():
                assert '#include "psad_half.cuh"' in ek.source and 'cuda_bf16' not in ek.source
                assert 'psad_bf16' in ek.source and 'psad_half ' not in ek.source
                key = ek.cache_key + '_spills'        # a key of its own: a cache hit would return no ptxas log
                _, log = runtime.compile_source(ek.source, key, list(ek.options) + ['--ptxas-options=-v'])
                os.remove(runtime.cubin_path(key))
                spills = [ln for ln in log.splitlines() if ln.startswith('ptxas') and 'spill' in ln]
                assert spills and all(' 0 bytes spill stores, 0 bytes spill loads' in ln for ln in spills), (variant, spills)


def test_bf16_march_geometry_and_cache_keys():
    import hashlib
    from pystencils_autodiff_b200 import emit as emit_mod
    ek = emit_march(configs.heat3d_op(shape=(8, 16, 128), dtype='bfloat16').forward_ast_gpu)
    # the 16-bit geometry of float16: 4 cells per lane, pads in 16-byte units, a box 128 + 2 x 8 cells wide
    assert ek.geometry['SX'] == 4 and ek.geometry['TX'] == 128
    assert [f['box'] for f in ek.plan['fields'] if f['tma']] == [(144, 34, 1)]
    assert all(f['elem_size'] == 2 for f in ek.plan['fields'])
    assert 'psad_lds_h4' in ek.source and 'psad_stg_h4' in ek.source and 'typedef psad_bf16' not in ek.source
    # fp32 kernels do not hash the 16-bit helpers; bf16 and fp16 kernels of the same stencil have keys of their own
    ek32 = emit_march(configs.heat3d_op(shape=(8, 16, 128)).forward_ast_gpu)
    h = hashlib.md5()
    h.update(emit_mod.EMITTER_VERSION.encode())
    h.update(ek32.source.encode())
    h.update(' '.join(ek32.options).encode())
    for fn in sorted(os.listdir(emit_mod.KERNEL_DIR)):
        if fn != 'psad_half.cuh':
            with open(os.path.join(emit_mod.KERNEL_DIR, fn), 'rb') as fh:
                h.update(fh.read())
    assert ek32.cache_key.endswith(h.hexdigest())
    ek16 = emit_march(configs.heat3d_op(shape=(8, 16, 128), dtype='float16').forward_ast_gpu)
    assert len({ek.cache_key, ek16.cache_key, ek32.cache_key}) == 3
    assert ek.source != ek16.source


def test_bf16_eligibility():
    import pystencils_autodiff_b200 as ps
    u = ps.fields('u: bfloat16[16,128]')
    lap = lambda o: [ps.Assignment(o.center, u[1, 0] + u[-1, 0] - 2 * u[0, 0])]     # noqa: E731
    for dt in ('float16', 'float32', 'float64'):
        op = ps.AutoDiffOp(lap(ps.fields('o: %s[16,128]' % dt)), op_name='mix', boundary_handling='zeros')
        assert march_ineligible_reason(op.forward_ast_gpu) == 'bfloat16 fields mixed with other field types', dt
    # float16 with a wider field keeps its own reason
    h = ps.fields('h: float16[16,128]')
    op = ps.AutoDiffOp([ps.Assignment(ps.fields('o: float32[16,128]').center, h[1, 0] - h[0, 0])], op_name='mix16')
    assert march_ineligible_reason(op.forward_ast_gpu) == 'float16 fields mixed with wider fields'
    assert march_ineligible_reason(configs.heat3d_op(shape=(4, 8, 128), dtype='bfloat16').forward_ast_gpu) is None


# ---- the march kernels on the CPU ----------------------------------------------------------------------------------------
@pytest.mark.timeout(600)
@pytest.mark.parametrize('make, shape, bh, which, tuning, scale', [
    (configs.heat3d_op, (9, 13, 136), 'zeros', 'forward', MarchTuning(ry=2, ty=6), 3e5),
    (configs.heat3d_op, (7, 11, 264), None, 'backward', MarchTuning(ry=1, ty=3, lookahead=1), 1e-9),
    (configs.heat3d_op, (5, 40, 136), 'zeros', 'backward', None, 1.0),            # the shipped geometry: 16+1 warps
    (configs.stencil27_op, (6, 9, 72), 'zeros', 'forward', MarchTuning(ry=3, ty=6), 1e6),
    (configs.stencil27_op, (5, 10, 136), None, 'backward', MarchTuning(ry=2, ty=4), 1.0),
    (configs.diffusion2d_op, (23, 136), 'zeros', 'forward', MarchTuning(ry=1, ty=4), 1e-10),
    (configs.diffusion2d_op, (21, 264), None, 'backward', MarchTuning(ry=1, ty=4), 1.0),
    (configs.tv_gradient_op, (3, 11, 136), 'zeros', 'forward', MarchTuning(ry=2, ty=4), 1.0),
    (configs.tv_gradient_op, (3, 9, 136), None, 'backward', MarchTuning(ry=1, ty=3), 1.0),
])
@pytest.mark.parametrize('full', [False, True])
def test_bf16_march_replay(make, shape, bh, which, tuning, scale, full):
    """The emitted march kernels with bf16 boxes: 8-byte shared loads widened into the fp32 register window, shuffled
    x-halos, packed bf16 stores; masked and mask-free instances, ragged y / z extents, magnitudes outside fp16's range.
    ``full``: under the real psad_march.cuh (TMA staging of 2-byte elements), else under the per-step shim."""
    op16, op64 = _ops(make, shape, bh)
    ir = op16.forward_ast_gpu if which == 'forward' else op16.backward_ast_gpu
    for masked in (True, False):
        if not masked and bh is None:
            continue          # 'none' boundary: the written cells reach beyond the iterated ones, only the masked instance
        ek = emit_march(ir, tuning, masked=masked)
        arrays, named = _inputs(ek, ir, shape, seed=3, scale=scale)
        if full:
            ctas, waits, loads = emu.run(ek, arrays, full=True, sm_count=2)
            assert ctas == 2 and loads > 0
        else:
            emu.run(ek, arrays)
        ref = _oracle(op64, which, named, bh)
        for f, a in zip(ek.fields, arrays):
            if f in ir.output_fields:
                got = from_words(a)
                assert not np.isnan(got).any()
                assert _rel_err(got, ref[f.name]) <= BF16_TOL, (f.name, masked, _rel_err(got, ref[f.name]))
                if scale != 1.0:
                    assert np.abs(ref[f.name]).max() > 1e5 or np.abs(ref[f.name]).max() < 1e-8


@pytest.mark.parametrize('which', ['forward', 'backward'])
def test_bf16_march_matches_generic(which):
    """The march kernel (plane sums, shared partial sums) and the generic kernel (one FMA chain per cell) evaluate the
    27-point sum in different orders: their bf16 results differ by at most one rounding step."""
    shape = (6, 18, 136)
    op16, _ = _ops(configs.stencil27_op, shape, 'zeros')
    ir = op16.forward_ast_gpu if which == 'forward' else op16.backward_ast_gpu
    ek = emit_march(ir, MarchTuning(ry=2, ty=6), masked=False)
    arrays, _ = _inputs(ek, ir, shape, seed=8)
    gen = emit_generic(ir)
    arrays_g = [a.copy() for a in arrays]
    emu.run(ek, arrays)
    emu.run_generic(gen, arrays_g)
    for f, a, b in zip(ek.fields, arrays, arrays_g):
        if f in ir.output_fields:
            assert _rel_err(from_words(a), from_words(b)) <= 2.0 ** -7
            assert np.mean(a != b) < 0.2
        else:
            assert np.array_equal(a, b)


# ---- generic kernels -----------------------------------------------------------------------------------------------------
def test_bf16_generic_strided_views_and_mixed_precision():
    import pystencils_autodiff_b200 as ps
    ex = lambda u_, o_: [ps.Assignment(o_.center, 0.5 * u_[0, 0] + 0.25 * u_[1, -2] - u_[-1, 1] * u_[0, 1])]   # noqa: E731
    u64, out64 = ps.fields('u, out: float64[9,14]')
    op64 = ps.AutoDiffOp(ex(u64, out64), op_name='strided64', boundary_handling='zeros')
    rng = np.random.default_rng(1)
    U = rng.uniform(-1, 1, (9, 14)) * 2e5
    Uw = np.asfortranarray(to_words(U))                                # x is NOT the contiguous axis
    ref = evaluate(op64.forward_assignments, {'u': from_words(np.ascontiguousarray(Uw))}, 'zeros')['out']
    u, out = ps.fields('u, out: bfloat16[9,14]')
    ek = emit_generic(ps.AutoDiffOp(ex(u, out), op_name='strided_bf', boundary_handling='zeros').forward_ast_gpu)
    assert 'typedef psad_bf16 T_0;' in ek.source and 'typedef float CT;' in ek.source
    big = np.full((9, 21), 0x7fc1, dtype=np.uint16)
    ot = big[:, 3:17]                                                  # row pitch 21 cells: unaligned rows
    emu.run_generic(ek, [ot, Uw])
    assert _rel_err(from_words(ot), ref) <= BF16_TOL
    assert np.all(big[:, :3] == 0x7fc1) and np.all(big[:, 17:] == 0x7fc1)
    # bf16 input, fp32 output (no output rounding to bf16), and fp32 input, bf16 output
    o32 = ps.fields('out: float32[9,14]')
    ir = ps.AutoDiffOp(ex(u, o32), op_name='mixed_bf', boundary_handling='zeros').forward_ast_gpu
    assert march_ineligible_reason(ir) == 'bfloat16 fields mixed with other field types' and ir.compute_dtype == np.float32
    O = np.full((9, 14), np.nan, dtype=np.float32)
    emu.run_generic(emit_generic(ir), [O, np.ascontiguousarray(Uw)])
    assert _rel_err(O.astype(np.float64), ref) <= 2e-6
    u32 = ps.fields('u: float32[9,14]')
    ir = ps.AutoDiffOp(ex(u32, out), op_name='mixed_bf2', boundary_handling='zeros').forward_ast_gpu
    W = np.full((9, 14), 0x7fc1, dtype=np.uint16)
    U32 = U.astype(np.float32)
    emu.run_generic(emit_generic(ir), [W, U32])
    ref32 = evaluate(op64.forward_assignments, {'u': U32.astype(np.float64)}, 'zeros')['out']
    assert _rel_err(from_words(W), ref32) <= BF16_TOL


def test_bf16_data_type_double():
    """``data_type='double'``: fp64 arithmetic on bf16 storage, one rounding from fp64 per cell."""
    from pystencils_autodiff_b200.ir import lower_assignments
    shape = (5, 12, 136)
    op16, op64 = _ops(configs.heat3d_op, shape, 'zeros')
    ir = lower_assignments(op16.forward_assignments, 'zeros', 'heat_d', data_type='double')
    assert ir.compute_dtype == np.float64
    for ek in (emit_march(ir, MarchTuning(ry=2, ty=6), masked=False), emit_generic(ir)):
        assert 'typedef double CT;' in ek.source
        arrays, named = _inputs(ek, ir, shape, seed=5, scale=1e-9)
        if ek.kind == 'march':
            emu.run(ek, arrays, full=True, sm_count=2)
        else:
            emu.run_generic(ek, arrays)
        ref = _oracle(op64, 'forward', named, 'zeros')['out']
        assert _rel_err(from_words(arrays[0]), ref) <= BF16_TOL


# ---- step decisions --------------------------------------------------------------------------------------------------------
def test_bf16_step_decisions():
    """TimeLoop default, fuse_steps=True, run_steps(fuse=True) and the unrolled slab Function agree: no fused bf16 pairs."""
    from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
    from pystencils_autodiff_b200.datahandling import SlabDataHandling, create_slab_unrolled_function
    for name, shape in (('c2', (8, 136)), ('c3', (8, 8, 136))):
        op = configs.make_config(name, shape=shape, dtype='bfloat16')
        k = CompiledKernel(op.forward_ast_gpu)
        assert k.fused_steps_reason() == FUSE_REASON
        with pytest.raises(ValueError, match=FUSE_REASON):
            k.emitted('march_x2')
        with pytest.raises(ValueError, match='bfloat16'):
            k.run_steps(torch.zeros(shape, dtype=torch.bfloat16), 4, fuse=True)
        for world, periodic, g in ((1, False, 0), (1, True, 2), (2, False, 2)):
            dh = SlabDataHandling(shape, 0, world, g, device='cpu', backend='torch', periodic=periodic)
            dh.add_arrays('u, out', dtype='bfloat16')
            for fuse in (None, True):
                tl = dh.create_timeloop(fuse_steps=fuse)
                tl.add_call(k, {})
                tl.swap('u', 'out')
                if fuse:
                    with pytest.raises(ValueError, match=FUSE_REASON):
                        tl.fused_pair()
                else:
                    assert tl.fused_pair() is None
            fn = create_slab_unrolled_function(op, dh, 4, fuse=None, kernel_class=CompiledKernel)
            assert fn.launches == [1] * 4
            with pytest.raises(ValueError, match=FUSE_REASON):
                create_slab_unrolled_function(op, dh, 4, fuse=True, kernel_class=CompiledKernel)


def test_bf16_run_steps_replayed():
    op16, op64 = _ops(configs.heat3d_op, (4, 16, 136), 'zeros')
    k = BF16Replay(op16.forward_ast_gpu)
    u0 = torch.from_numpy(np.random.default_rng(2).uniform(-1, 1, (4, 16, 136))).to(torch.bfloat16)
    ReplayKernel.launches.clear()
    out = k.run_steps(u0, 3)
    assert out.dtype == torch.bfloat16
    assert ReplayKernel.launches == ['psad_heat3d_forward_gpu_march_nomask'] * 3
    assert _rel_err(out.double().numpy(), _rounded_steps(op64, u0.double().numpy(), 3, 'zeros')) <= STEPS_TOL


class _StubPeer:
    """Stands in for the CUDA IPC machinery: records what would be registered."""

    def __init__(self, dh):
        self.registered = []

    def register(self, t):
        self.registered.append(t)

    def close(self):
        pass


def _glob_u(world):
    gshape = (5 * world, 14, 136)
    return torch.from_numpy(np.random.default_rng(7).uniform(-1, 1, gshape)).to(torch.bfloat16)


def _slab_worker(rank, world, port, steps, q, shim_root):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    use_bf16_shims(shim_root)
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from pystencils_autodiff_b200 import datahandling
        from pystencils_autodiff_b200.datahandling import SlabDataHandling
        glob_u = _glob_u(world)
        res = {}
        for bh in ('zeros', None):
            dh = SlabDataHandling(tuple(glob_u.shape), rank, world, 1, device='cpu', backend='torch')
            dh.add_arrays('u, out', dtype='bfloat16')
            op_l = configs.heat3d_op(shape=dh.dec.local_shape, dtype='bfloat16', boundary_handling=bh)
            kernel = BF16Replay(op_l.forward_ast_gpu)
            dh.owned('u').copy_(glob_u[dh.dec.start:dh.dec.start + dh.dec.n_local])
            ReplayKernel.launches.clear()
            tl = dh.create_timeloop()
            tl.add_call(kernel, {'halo_fields': ['u']})
            tl.swap('u', 'out')
            tl.run(steps)
            assert not tl.fused_last_run
            parts = 1 + int(rank > 0) + int(rank < world - 1)
            assert len(ReplayKernel.launches) == parts * steps and all('march' in n for n in ReplayKernel.launches)
            res[bh] = dh.gather_array('u')
        # peer halos: refused outright for bfloat16 arrays
        orig = datahandling._PeerHalo
        datahandling._PeerHalo = _StubPeer
        try:
            dh = SlabDataHandling(tuple(glob_u.shape), rank, world, 1, device='cpu', backend='torch', peer_halo=True)
            assert dh.peer is not None
            dh.add_array('a32', dtype=np.float32)
            try:
                dh.add_array('abf', dtype='bfloat16')
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
def test_bf16_slab_time_loop_two_ranks(_bf16_shims):
    """Two gloo ranks, ghost planes exchanged as bf16, single-step TimeLoop on the replayed march kernels against the
    step-by-step oracle rounded to bf16 after every step; ``peer_halo=True`` refuses bfloat16 arrays."""
    world, steps = 2, 3
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29160                     # outside the ranges the other multi-process tests draw from
    procs = [ctx.Process(target=_slab_worker, args=(r, world, port, steps, q, str(_bf16_shims)))
             for r in range(world)]
    for p in procs:
        p.start()
    import test_slab_gloo
    results = test_slab_gloo._collect(procs, q, world)
    glob_u = _glob_u(world)
    for bh in ('zeros', None):
        op64 = configs.heat3d_op(shape=tuple(glob_u.shape), dtype='float64', boundary_handling=bh)
        ref = _rounded_steps(op64, glob_u.double().numpy(), steps, bh)
        for rank, res, peer_error in results:
            assert res[bh].dtype == np.float32           # gather_array widens bf16 to float32
            assert _rel_err(res[bh].astype(np.float64), ref) <= STEPS_TOL, (bh, rank)
            assert peer_error is not None and 'bfloat16' in peer_error
