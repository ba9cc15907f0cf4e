"""The random stencils of tests/stencil_fuzz.py in float16 and bfloat16 on the CPU, checked cell by cell against the fp64
oracle (``stencil_fuzz.check_cells``): x-halos of 1-4 cells, asymmetric halos, several input fields with different pads,
several outputs, non-linear terms, both boundary modes, ghost layers that are not a multiple of 4.  The march kernels
(masked with a launch range whose x bounds cut inside a lane, and the instance a plain launch takes) are replayed by
``march_emulator.run``, the generic kernel by ``march_emulator.run_generic``; bfloat16 under the host stand-ins of
tests/test_bf16_replay.py.  The same cases run on the GPU in tests/test_gpu_fuzz16.py.

The per-cell bound is half a spacing of the stored type plus the fp32 allowance, so a store that rounds the wrong way, a
flushed subnormal or a double rounding under ``data_type='double'`` fails where the norm-wise 5e-4 / 4e-3 of
tests/test_half_replay.py and tests/test_bf16_replay.py can pass.  A subset of the seeds keeps the file to about a minute:
every feature above is in it."""
import numpy as np
import pytest

import march_emulator as emu
from oracle.evaluate import evaluate
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
from stencil_fuzz import (DOUBLE_SHAPES, KAPPA_DOUBLE, SCALED, check_outputs, fuzz_case, fuzz_inputs, ragged_range,
                          reached)
from test_bf16_replay import use_bf16_shims

# 1: 2-D, x-halo 4, three inputs, ghost layers 4, ragged 136; 9: 3-D, x 40 (one partial tile), ghost layers 2;
# 6: 3-D 'zeros', three inputs, two outputs; 15: 2-D, ghost layers 3; 23: 3-D, ghost layers 1, x 40;
# 18: 2-D 'zeros', x 264; 5: 3-D, ghost layers 3, the extent grown from 5 to 9 planes
SEEDS = [1, 9, 6, 15, 23, 18, 5]


@pytest.fixture(scope='module', autouse=True)
def _bf16_shims(tmp_path_factory):
    with pytest.MonkeyPatch.context() as mp_:
        use_bf16_shims(tmp_path_factory.mktemp('bf16_shims'), mp_)
        yield


def _replay(ek, stored, launch_range=None):
    arrays = []
    for f in ek.fields:
        a = emu.aligned_empty(stored[f.name].shape, stored[f.name].dtype)
        a[...] = stored[f.name]
        arrays.append(a)
    if ek.kind == 'march':
        emu.run(ek, arrays, launch_range=launch_range)
    else:
        emu.run_generic(ek, arrays, launch_range=launch_range)
    return {f.name: a for f, a in zip(ek.fields, arrays)}


def _instances(ir, shape, march=True):
    """``(name, emitted kernel, launch range)`` of the instances CompiledKernel launches for dense arrays of ``shape``."""
    k = CompiledKernel(ir)
    out = [('generic', k._emitted['generic'], None)]
    if march and 'march' in k._emitted and shape[-1] * 2 % 16 == 0:
        out.append(('march+range', k._emitted['march'], ragged_range(shape, ir.ghost_layers)))
        plain = 'march_nomask' if ir.boundary == 'zeros' or ir.ghost_layers == 0 else 'march'
        out.append((plain, k._emitted[plain], None))
    return out


def _run_case(seed, kernels, shape, bh, which=(0, 1), diff_scale=1.0, kappa=None, march=True):
    """Replays the kernels ``which`` of the case on every instance, checks them; returns the oracle results."""
    kw = {} if kappa is None else dict(kappa=kappa)
    refs = []
    for i in which:
        ir, assigns = kernels[i]
        stored, values = fuzz_inputs(ir.all_fields, ir, shape, seed, diff_scale)
        ref = evaluate(assigns, values, bh)
        for name, ek, rng in _instances(ir, shape, march):
            got = _replay(ek, stored, rng)
            check_outputs(ir, got, ref, rng, floor=diff_scale, what='seed %d %s %s' % (seed, ir.function_name, name), **kw)
        refs += [ref[f.name] for f in ir.output_fields]
    return refs


@pytest.mark.timeout(600)
@pytest.mark.parametrize('seed', SEEDS)
@pytest.mark.parametrize('dtype', ['float16', 'bfloat16'])
def test_lowp_random_stencils_replay(dtype, seed):
    op, kernels, bh, shape = fuzz_case(seed, dtype)
    _run_case(seed, kernels, shape, bh)


@pytest.mark.timeout(600)
@pytest.mark.parametrize('dtype, seed, scale', SCALED)
def test_lowp_random_stencils_scaled_replay(dtype, seed, scale):
    op, kernels, bh, shape = fuzz_case(seed, dtype)
    reached(dtype, scale, _run_case(seed, kernels, shape, bh, which=(1,), diff_scale=scale))


@pytest.mark.timeout(600)
@pytest.mark.parametrize('dtype, seed', [('float16', 6), ('bfloat16', 1)])
def test_lowp_random_stencils_double_replay(dtype, seed):
    """``data_type='double'``: fp64 arithmetic, each stored cell rounded once from fp64 (κ = 1e-12: a rounding through
    fp32 fails, ``DOUBLE_SHAPES``).  The generic kernel only: the march kernels replayed at this size would take minutes;
    tests/test_gpu_fuzz16.py runs them."""
    shape = DOUBLE_SHAPES[len(fuzz_case(seed, dtype)[3])]
    op, kernels, bh, shape = fuzz_case(seed, dtype, shape=shape, data_type='double')
    assert op.forward_ast_gpu.compute_dtype == np.float64
    _run_case(seed, kernels, shape, bh, which=(0,), kappa=KAPPA_DOUBLE, march=False)


@pytest.mark.parametrize('seed', [6, 15, 21])
def test_mixed_type_random_stencils_replay(seed):
    """Each field its own type of float16, bfloat16 and float32: the generic kernel, each output checked in its type."""
    op, kernels, bh, shape = fuzz_case(seed, mixed=True)
    assert 'march' not in CompiledKernel(op.forward_ast_gpu)._emitted
    _run_case(seed, kernels, shape, bh)
