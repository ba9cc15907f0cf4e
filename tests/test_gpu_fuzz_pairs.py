"""GPU: fused pairs of steps (emit_chain.py, ``out = S(S(u))`` in one launch: TMA ring, mbarriers, rows exchanged between
warps or recomputed) on the random one-field stencils of ``stencil_fuzz.random_pair_stencil`` — the pair kernel against
the fp64 oracle applied twice, ``run_steps`` against the oracle and single steps (and single steps only where no pair can
be built), slab launches of the pair against the whole-array launch.  CPU replay of the same stencils:
tests/test_pair_fuzz_replay.py."""
import numpy as np
import pytest

from pystencils_autodiff_b200 import runtime
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
from pystencils_autodiff_b200.emit import MarchTuning
from stencil_fuzz import PAIR_SEEDS, WIDE_TOL, check_steps, oracle_steps, pair_case, pair_input

pytestmark = pytest.mark.gpu

ROW_MODES = {'exchanged': None, 'recomputed': MarchTuning(exchange=False)}
STEPS = (2, 3, 5)
# 3-D seeds whose forward pair runs on two emulated slabs: fp64 / boundary None, fp32 / 'zeros' with a scalar, fp32 /
# boundary None with z reach 2 and fix-up loads
SLAB_SEEDS = (6, 8, 30)
SLAB_PLANES, SLAB_WORLD = 8, 2


def _launches():
    """Native kernel launches so far (in the CPU dry run of these bodies, tests/dryrun_plugin.py: replayed launches)."""
    return runtime.launch_count() + len(getattr(CompiledKernel, 'launches', ()))


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def pair_kernel(ir, tuning):
    k = CompiledKernel(ir)
    k.tuning_x2 = tuning
    return k


@pytest.mark.parametrize('seed', PAIR_SEEDS)
def test_random_pair_matches_oracle_twice(seed):
    """One pair launch on a NaN-prefilled output == the oracle applied twice, both row modes, forward and adjoint; the
    input is not touched.  A stencil without any pair runs one single step against the oracle instead."""
    import torch
    kernels, bh, shape, dtype, scalars = pair_case(seed)
    u = pair_input(shape, dtype, seed)
    ut = _t(u)
    pairs = 0
    for which, ir, assigns in kernels:
        fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
        ref = oracle_steps(assigns, ir, u, 2, bh, scalars)
        for mode, tuning in ROW_MODES.items():
            k = pair_kernel(ir, tuning)
            if k.fused_steps_reason():
                continue
            out = torch.full_like(ut, float('nan'))
            k(**{fin: ut, fout: out}, _variant='march_x2', **scalars)
            assert k.last_instance == 'march_x2'
            check_steps(out.cpu().numpy(), ref, dtype, (seed, which, mode))
            assert torch.equal(ut, _t(u)), (seed, which, mode, 'the input was written')
            pairs += 1
    if not pairs:
        which, ir, assigns = kernels[0]
        k = CompiledKernel(ir)
        out = torch.full_like(ut, float('nan'))
        k(**{ir.input_fields[0].name: ut, ir.output_fields[0].name: out}, **scalars)
        check_steps(out.cpu().numpy(), oracle_steps(assigns, ir, u, 1, bh, scalars), dtype, (seed, which, 'one step'))


@pytest.mark.parametrize('seed', PAIR_SEEDS)
def test_random_pair_run_steps(seed):
    """``run_steps(u, T)``: T // 2 pair launches + T % 2 single ones where a pair can be built, else T single launches
    (never an error); against the oracle applied T times and against ``fuse=False`` (bit for bit without pairs)."""
    import torch
    kernels, bh, shape, dtype, scalars = pair_case(seed)
    u = pair_input(shape, dtype, seed)
    ut = _t(u)
    for which, ir, assigns in kernels:
        k = CompiledKernel(ir)
        pair = k.fused_steps_reason() is None
        for steps in STEPS:
            what = (seed, which, steps)
            n0 = _launches()
            fused = k.run_steps(ut, steps, **scalars)
            assert _launches() - n0 == (steps // 2 + steps % 2 if pair else steps), what
            n0 = _launches()
            single = k.run_steps(ut, steps, fuse=False, **scalars)
            assert _launches() - n0 == steps, what
            ref = oracle_steps(assigns, ir, u, steps, bh, scalars)
            check_steps(fused.cpu().numpy(), ref, dtype, what)
            check_steps(single.cpu().numpy(), ref, dtype, what + ('fuse=False',))
            if pair:
                scale = max(1.0, np.abs(ref).max())
                assert (fused - single).abs().max().item() <= WIDE_TOL[dtype] * scale, what
            else:
                assert torch.equal(fused, single), what
        assert torch.equal(ut, _t(u)), (seed, which, 'the input was written')


def slab_case(seed):
    """``pair_case`` of ``seed`` with ``SLAB_WORLD`` slabs of ``SLAB_PLANES`` planes along z, and the reach ``g`` of
    its forward kernel along z."""
    shape = (SLAB_WORLD * SLAB_PLANES,) + pair_case(seed)[2][1:]
    case = pair_case(seed, shape)
    ir = case[0][0][1]
    return case, max(ir.halo(ir.input_fields[0].name)[0])


def slab_local_kernel(seed, g):
    """The forward kernel of ``seed`` on one slab with its ``2 g`` ghost planes per side."""
    shape = (SLAB_PLANES + 4 * g,) + pair_case(seed)[2][1:]
    return CompiledKernel(pair_case(seed, shape)[0][0][1])


@pytest.mark.parametrize('seed', SLAB_SEEDS)
def test_random_pair_slab_launches_match_whole_array(seed):
    """The pair on slabs: every rank's interior / boundary launches (``datahandling.slab_ranges(..., steps=2)``) over its
    slab with ``2 g`` ghost planes copied in reproduce the whole-array pair launch bit for bit; ghost planes stay
    unwritten."""
    import torch
    from pystencils_autodiff_b200.datahandling import slab_ranges
    (kernels, bh, shape, dtype, scalars), g = slab_case(seed)
    which, ir, assigns = kernels[0]
    k = CompiledKernel(ir)
    assert g > 0 and k.fused_steps_reason() is None
    fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
    u = pair_input(shape, dtype, seed)
    whole = torch.full(shape, float('nan'), dtype=getattr(torch, dtype), device='cuda')
    k(**{fin: _t(u), fout: whole}, _variant='march_x2', **scalars)
    whole = whole.cpu().numpy()
    check_steps(whole, oracle_steps(assigns, ir, u, 2, bh, scalars), dtype, (seed, 'whole array'))
    n, G = SLAB_PLANES, 2 * g
    local_k = slab_local_kernel(seed, g)
    for rank in range(SLAB_WORLD):
        start = rank * n
        local_u = np.zeros((n + 2 * G,) + shape[1:], dtype=dtype)
        lo, hi = max(0, start - G), min(shape[0], start + n + G)
        local_u[lo - (start - G):hi - (start - G)] = u[lo:hi]        # owned planes + received ghost planes
        local_t = _t(local_u)
        local_out = torch.full(local_u.shape, float('nan'), dtype=getattr(torch, dtype), device='cuda')
        parts = slab_ranges(shape, start, n, G, rank > 0, rank < SLAB_WORLD - 1, 'zeros' if bh == 'zeros' else 'none',
                            ir.ghost_layers, 3, steps=2, halo=g)
        for part in parts:
            if part is not None:
                local_k(**{fin: local_t, fout: local_out}, _variant='march_x2', _range=part, **scalars)
        local_out = local_out.cpu().numpy()
        assert np.array_equal(local_out[G:G + n], whole[start:start + n]), (seed, rank)
        assert np.isnan(local_out[:G]).all() and np.isnan(local_out[G + n:]).all(), (seed, rank, 'ghost planes written')
