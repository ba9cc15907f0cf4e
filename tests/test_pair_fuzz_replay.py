"""Fused pairs of steps (emit_chain.py, ``out = S(S(u))`` in one launch) on the random one-field stencils of
``stencil_fuzz.random_pair_stencil``, replayed on the CPU (tests/march_emulator.py) against the fp64 oracle applied
twice — both ways of getting the intermediate rows of the neighbouring warps (exchanged, recomputed), forward and
adjoint — and the rule that a stencil whose pair cannot be built takes single steps.  The same stencils run on the GPU
in tests/test_gpu_fuzz_pairs.py."""
import functools
import re

import numpy as np
import pytest
import sympy as sp

import march_emulator as emu
import pystencils_autodiff_b200 as ps
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
from pystencils_autodiff_b200.emit import MarchTuning
from pystencils_autodiff_b200.emit_chain import chain_ineligible_reason, emit_march_chain
from stencil_fuzz import PAIR_SEEDS, check_steps, oracle_steps, pair_case, pair_input

ROW_MODES = {'exchanged': None, 'recomputed': MarchTuning(exchange=False)}


def pair_kernel(ir, tuning):
    k = CompiledKernel(ir)
    k.tuning_x2 = tuning
    return k


def replay_pair(k, u, scalars, full=False):
    """``out = S(S(u))`` through the CPU replay of ``k``'s pair kernel, on a NaN-prefilled output; the input must come
    back untouched."""
    ek = k.emitted('march_x2')
    fout = k.ir.output_fields[0].name
    src = emu.aligned_empty(u.shape, u.dtype)
    src[...] = u
    out = emu.aligned_empty(u.shape, u.dtype, np.nan)
    arrays = [out if f.name == fout else src for f in ek.fields]
    if u.ndim == 2:                     # the lifted pair takes one-plane 3-D fields (CompiledKernel.__call__)
        arrays = [a[None] for a in arrays]
    emu.run(ek, arrays, [scalars[s] for s in ek.scalars], full=full)
    assert np.array_equal(src, u), 'the input was written'
    return out


@functools.lru_cache(maxsize=None)
def profile(seed):
    """What seed ``seed`` exercises: stencil features, and per (direction, row mode) the pair's reason / geometry."""
    kernels, bh, shape, dtype, scalars = pair_case(seed)
    ir = kernels[0][1]
    p = dict(ndim=len(shape), dtype=dtype, bh=bh, shape=shape, scalar=bool(scalars), halo=ir.halo('u'),
             constant=any(not t.atoms(ps.Field.Access) for t in sp.Add.make_args(sp.expand(ir.main[0][1]))),
             nonlinear=len(kernels) == 1,          # the adjoint of a non-linear stencil reads u too: no one-field kernel
             pairs={})
    for which, kir, _ in kernels:
        for mode, tuning in ROW_MODES.items():
            k = pair_kernel(kir, tuning)
            reason = k.fused_steps_reason()
            p['pairs'][which, mode] = reason if reason else k.emitted('march_x2')
    return p


def test_pair_seeds_cover_the_features():
    """The seed list exercises every feature the pair emitter has code for, several times over, so that an edit of the
    generator cannot silently drop one."""
    counts = {}

    def count(feature, n=1):
        counts[feature] = counts.get(feature, 0) + n

    for seed in PAIR_SEEDS:
        p = profile(seed)
        count(('%d-D' % p['ndim']))
        count(p['dtype'])
        count('boundary %s' % p['bh'])
        count('scalar', p['scalar'])
        count('access-free term', p['constant'])
        count('non-linear', p['nonlinear'])
        count('one-sided', any((lo == 0) != (hi == 0) for lo, hi in p['halo']))
        count('z reach 2', p['ndim'] == 3 and max(p['halo'][0]) == 2)
        count('asymmetric z reach', p['ndim'] == 3 and p['halo'][0][0] != p['halo'][0][1])
        fwd = p['pairs']['forward', 'exchanged']
        if isinstance(fwd, str):
            count('no pair (x reach wider than a strip)', 'wider than the per-thread strip' in fwd)
            continue
        count('adjoint pair', ('adjoint', 'exchanged') in p['pairs'])
        fix = 'if (lane == 0)' in fwd.source or 'if (lane == 31)' in fwd.source
        count('fix-up loads %s' % p['dtype'], fix)
        count('x reach filling two radii of a strip', not fix and 2 * max(p['halo'][-1]) == fwd.geometry['SX'])
        count('rows exchanged', fwd.geometry['exchange'])
        count('rows recomputed (default)', not fwd.geometry['exchange'])
        count('y below one tile', p['shape'][-2] < fwd.plan['tile_y'])
        count('y above one tile', p['shape'][-2] > fwd.plan['tile_y'])
        assert p['shape'][-1] > fwd.plan['tile_x'], (seed, 'x spans more than one tile')
        if p['ndim'] == 3:
            count('z below the warm-up', p['shape'][0] < fwd.plan['warmup'])
            count('z above the warm-up', p['shape'][0] > fwd.plan['warmup'])
    print(counts)
    for feature in ('2-D', '3-D', 'float32', 'float64', 'boundary zeros', 'boundary None', 'scalar', 'access-free term',
                    'non-linear', 'one-sided', 'z reach 2', 'asymmetric z reach', 'no pair (x reach wider than a strip)',
                    'adjoint pair', 'fix-up loads float32', 'fix-up loads float64', 'x reach filling two radii of a strip',
                    'rows exchanged', 'rows recomputed (default)', 'y below one tile', 'y above one tile',
                    'z below the warm-up', 'z above the warm-up'):
        assert counts.get(feature, 0) >= 3, (feature, counts.get(feature, 0))


def test_fused_steps_reason_is_the_emitters():
    """``CompiledKernel.fused_steps_reason()`` is None exactly when the pair can be emitted with the kernel's tuning, and
    the form check alone (``chain_ineligible_reason``) already refuses what the emitter's x strip cannot hold."""
    for seed in PAIR_SEEDS:
        for which, ir, _ in pair_case(seed)[0]:
            chain_ir = CompiledKernel(ir)._chain_ir()
            for mode, tuning in ROW_MODES.items():
                got = profile(seed)['pairs'][which, mode]
                try:
                    emit_march_chain(chain_ir, tuning)
                    error = None
                except ValueError as e:
                    error = str(e)
                assert isinstance(got, str) == (error is not None), (seed, which, mode, got, error)
                form = chain_ineligible_reason(chain_ir, tuning)
                assert (form is None) == (error is None), (seed, which, mode, form, error)


@pytest.mark.timeout(300)
@pytest.mark.parametrize('seed', PAIR_SEEDS)
def test_random_pair_replay(seed):
    """``S(S(u))`` from one pair launch == the oracle applied twice, both row modes, forward and adjoint."""
    kernels, bh, shape, dtype, scalars = pair_case(seed)
    u = pair_input(shape, dtype, seed)
    for which, ir, assigns in kernels:
        ref = oracle_steps(assigns, ir, u, 2, bh, scalars)
        for mode, tuning in ROW_MODES.items():
            k = pair_kernel(ir, tuning)
            if k.fused_steps_reason():
                continue
            check_steps(replay_pair(k, u, scalars), ref, dtype, (seed, which, mode))


# seeds through the real psad_march.cuh (producer warp, TMA ring, mbarriers; tests/cpu_shim_full): fp32 with fix-up loads
# and exchanged rows, a lifted 2-D fp64 stencil with fix-up loads, fp64 boundary None with exchanged rows and a scalar
FULL_SEEDS = (0, 7, 21)


@pytest.mark.timeout(600)
@pytest.mark.parametrize('seed', FULL_SEEDS)
def test_random_pair_full_pipeline_replay(seed):
    kernels, bh, shape, dtype, scalars = pair_case(seed)
    which, ir, assigns = kernels[0]
    u = pair_input(shape, dtype, seed)
    k = pair_kernel(ir, None)
    assert k.fused_steps_reason() is None
    check_steps(replay_pair(k, u, scalars, full=True), oracle_steps(assigns, ir, u, 2, bh, scalars), dtype, (seed, which))


# parts of an emitted pair kernel the replay must depend on: the pad-column loads of the row's edge lanes (x reach beyond
# half a strip), the select that forces the intermediate field to 0 outside the iteration range (what the second of two
# launches reads there), and the barrier after which the warps read each other's intermediate rows
MUTATIONS = {
    'fix-up loads': lambda s: re.subn(r'\n  if \(lane == (?:0|31)\) u\d+\[\d+\] = p\d+\[-?\d+\];', '', s),
    'zero-forcing select': lambda s: re.subn(r'\n    t\d+\[\d+\] = \(\(\(tm >> \d+\) & 1u\) && .*? : \(CT\)0;', '', s),
    'consumer barrier': lambda s: re.subn(r'\n  psad_consumer_barrier\(cfg::THREADS\);', '', s),
}


@pytest.mark.parametrize('mutation', sorted(MUTATIONS))
def test_replay_detects_a_mutated_pair_kernel(mutation):
    """The first seed whose forward pair (rows exchanged) has the part fails its check once the part is removed."""
    for seed in PAIR_SEEDS:
        kernels, bh, shape, dtype, scalars = pair_case(seed)
        which, ir, assigns = kernels[0]
        k = pair_kernel(ir, None)
        if k.fused_steps_reason():
            continue
        ek = k.emitted('march_x2')
        source, n = MUTATIONS[mutation](ek.source)
        if n:
            break
    else:
        pytest.fail('no seed has %s' % mutation)
    ek.source = source
    u = pair_input(shape, dtype, seed)
    with pytest.raises(AssertionError):
        check_steps(replay_pair(k, u, scalars), oracle_steps(assigns, ir, u, 2, bh, scalars), dtype, (seed, mutation))


def test_wide_x_reach_takes_single_steps():
    """An fp64 stencil reaching 3 cells along x (fp64 strips are 2 cells) has no pair: ``fused_steps_reason`` says so, and
    everything that takes pairs by default runs single steps instead of failing at the first launch."""
    import torch
    from pystencils_autodiff_b200.datahandling import SlabDataHandling, SlabDecomposition, _fused_pair_reason
    from replay_kernels import ReplayKernel
    shape = (9, 24, 128)
    u, out = ps.fields('u, out: float64[%d,%d,%d]' % shape)
    rhs = 0.5 * u[0, 0, 0] + 0.25 * u[0, 0, 3] + 0.25 * u[0, 0, -1]
    x = pair_input(shape, 'float64', 3)
    for bh in ('zeros', None):
        op = ps.AutoDiffOp(ps.AssignmentCollection([ps.Assignment(out.center, rhs)]), op_name='wide', boundary_handling=bh)
        for ir, assigns in ((op.forward_ast_gpu, op.forward_assignments), (op.backward_ast_gpu, op.backward_assignments)):
            k = ReplayKernel(ir)
            ReplayKernel.launches = []
            got = k.run_steps(torch.from_numpy(x), 3)
            assert len(ReplayKernel.launches) == 3 and not any('x2' in n for n in ReplayKernel.launches)
            ref = oracle_steps(assigns, ir, x, 3, bh, {})
            assert np.abs(got.numpy() - ref).max() <= 1e-13
            if ir is op.forward_ast_gpu:       # the data handling's time loop (one rank, no ghost planes)
                dh = SlabDataHandling(shape, 0, 1, 0, device='cpu', backend='torch')
                dh.add_arrays('u, out', dtype=np.float64)
                dh.gpu_arrays['u'].copy_(torch.from_numpy(x))
                ReplayKernel.launches = []
                dh.run_steps(k, 3)
                assert len(ReplayKernel.launches) == 3 and not any('x2' in n for n in ReplayKernel.launches)
                assert np.array_equal(dh.gpu_arrays['u'].numpy(), got.numpy())
            assert 'wider than the per-thread strip' in k.fused_steps_reason()
            assert 'wider than the per-thread strip' in chain_ineligible_reason(ir)
            assert 'wider than the per-thread strip' in _fused_pair_reason(k, SlabDecomposition(shape, 0, 1, 0))
            with pytest.raises(ValueError, match='wider than the per-thread strip'):
                k.emitted('march_x2')
            with pytest.raises(ValueError, match='wider than the per-thread strip'):
                k.run_steps(torch.from_numpy(x), 2, fuse=True)
    # a strip that holds the reach (sx=4 for fp64) gives the pair back
    from pystencils_autodiff_b200.emit import MarchTuning as T
    assert chain_ineligible_reason(op.forward_ast_gpu, T(sx=4)) is None
    assert emit_march_chain(op.forward_ast_gpu, T(sx=4)).geometry['SX'] == 4
