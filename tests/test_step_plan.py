"""When do fused pairs of steps run on a slab data handling?  The default (``fuse_steps=None`` / ``fuse=None``) and an
explicit request (``fuse_steps=True``) must agree with each other and with what ``run_kernel(..., fused_steps=2)``
accepts, for every entry point that decides it.  Host logic only: no process group, no kernel launch."""
import itertools

import numpy as np
import pytest

from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
from pystencils_autodiff_b200.configs import make_config
from pystencils_autodiff_b200.datahandling import SlabDataHandling, create_slab_unrolled_function

_SHAPES = {'c2': (8, 136), 'c3': (8, 8, 136)}


def _expected_pairs(name, world, periodic, g, dtype):
    if dtype == 'float16':
        return False                       # fused pairs are not implemented for float16 fields
    if name == 'c2':
        return world == 1 and g == 0       # 2-D pairs run on whole arrays only
    return (world == 1 and not periodic) or g >= 2        # 3-D: ghost planes for twice the reach (1 plane)


@pytest.mark.parametrize('name', sorted(_SHAPES))
def test_fused_pair_decisions_agree(name):
    shape = _SHAPES[name]
    ops = {dt: make_config(name, shape=shape, dtype=dt) for dt in ('float32', 'float16')}
    kernels = {dt: CompiledKernel(op.forward_ast_gpu) for dt, op in ops.items()}
    for world, periodic, g, dt in itertools.product((1, 2), (False, True), (0, 1, 2), ('float32', 'float16')):
        case = (name, world, periodic, g, dt)
        expected = _expected_pairs(*case)
        dh = SlabDataHandling(shape, 0, world, g, device='cpu', backend='torch', periodic=periodic)
        dh.add_arrays('u, out', dtype=np.dtype(dt))
        loops = {}
        for fuse in (None, True):
            loops[fuse] = dh.create_timeloop(fuse_steps=fuse)
            loops[fuse].add_call(kernels[dt], {})
            loops[fuse].swap('u', 'out')
        by_default = loops[None].fused_pair() is not None
        try:
            loops[True].fused_pair()
            on_request = True
        except ValueError:
            on_request = False
        assert by_default == on_request == expected, case
        # the unrolled slab Function: sharded slabs need ghost planes for one step even when no pair runs
        sharded = world > 1 or periodic
        try:
            fn = create_slab_unrolled_function(ops[dt], dh, 4, fuse=None, kernel_class=CompiledKernel)
        except ValueError as e:
            assert sharded and g == 0 and 'ghost layers' in str(e), case
            continue
        assert (2 in fn.launches) == expected, (case, fn.launches)
