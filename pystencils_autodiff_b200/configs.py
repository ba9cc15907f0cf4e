"""The five stencils of ``BASELINE.json`` (SURVEY.md §8d) as ``AutoDiffOp`` factories.

Shared by ``bench.py``, ``__graft_entry__.py`` and the tests so that all of them run exactly the same operators.
Shapes and dtypes are parameters: the benchmark uses the full sizes, the parity tests small ones.
"""
import itertools

import sympy as sp

from ._autodiff import AutoDiffOp
from .assignment import Assignment, AssignmentCollection
from .field import fields

__all__ = ['readme_op', 'diffusion2d_op', 'heat3d_op', 'stencil27_op', 'tv_gradient_op', 'CONFIG_SHAPES', 'make_config']

_DT = {'bfloat16': 'bfloat16', 'float16': 'float16', 'float32': 'float32', 'float64': 'float64'}


def _shape_str(shape):
    return ','.join(str(int(s)) for s in shape)


def readme_op(shape=(20, 30), dtype='float32', boundary_handling=None, **kw):
    """C1 — README example ``z = x*log(x*y)`` (/root/reference/README.rst:55-59)."""
    z, y, x = fields('z, y, x: %s[%s]' % (_DT[dtype], _shape_str(shape)))
    fa = AssignmentCollection({z[0, 0]: x[0, 0] * sp.log(x[0, 0] * y[0, 0])})
    return AutoDiffOp(fa, op_name='readme', boundary_handling=boundary_handling, **kw)


def diffusion2d_op(shape=(8192, 8192), dtype='float32', alpha=0.1, boundary_handling='zeros', **kw):
    """C2 — 2-D 5-point diffusion step ``out = u + alpha*(u_N + u_S + u_E + u_W - 4u)``."""
    u, out = fields('u, out: %s[%s]' % (_DT[dtype], _shape_str(shape)))
    rhs = u[0, 0] + alpha * (u[1, 0] + u[-1, 0] + u[0, 1] + u[0, -1] - 4 * u[0, 0])
    return AutoDiffOp([Assignment(out.center, rhs)], op_name='diffusion2d', boundary_handling=boundary_handling, **kw)


def heat3d_op(shape=(1024, 1024, 1024), dtype='float32', alpha=0.1, boundary_handling='zeros', **kw):
    """C3 — 3-D 7-point heat-equation step."""
    u, out = fields('u, out: %s[%s]' % (_DT[dtype], _shape_str(shape)))
    nb = sum(u[o] for o in [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)])
    rhs = u[0, 0, 0] + alpha * (nb - 6 * u[0, 0, 0])
    return AutoDiffOp([Assignment(out.center, rhs)], op_name='heat3d', boundary_handling=boundary_handling, **kw)


def stencil27_op(shape=(768, 768, 768), dtype='float64', weights=(0.4, 0.05, 0.02, 0.0075),
                 boundary_handling='zeros', **kw):
    """C4 — 3-D 27-point stencil, one weight per neighbour class (centre, 6 faces, 12 edges, 8 corners)."""
    u, out = fields('u, out: %s[%s]' % (_DT[dtype], _shape_str(shape)))
    classes = {0: 0, 1: 0, 2: 0, 3: 0}
    for o in itertools.product((-1, 0, 1), repeat=3):
        classes[sum(abs(v) for v in o)] += u[o]
    rhs = sum(sp.Float(w) * classes[k] for k, w in enumerate(weights))
    return AutoDiffOp([Assignment(out.center, rhs)], op_name='stencil27', boundary_handling=boundary_handling, **kw)


def tv_gradient_op(shape=(16, 4096, 4096), dtype='float32', lam=1.0, eps=1e-3, boundary_handling='zeros', **kw):
    """C5 — total-variation denoising gradient on a batch of images (zero offsets along dim 0):
    ``g = lam*(u - f) - div(grad u / sqrt(|grad u|^2 + eps^2))`` with forward differences for the gradient and
    backward differences for the divergence."""
    u, f, g = fields('u, f, g: %s[%s]' % (_DT[dtype], _shape_str(shape)))
    e2 = sp.Float(eps) ** 2

    def U(dy, dx):
        return u[0, dy, dx]

    def flux(dy, dx):  # (px, py) at the cell shifted by (dy, dx)
        ux = U(dy, dx + 1) - U(dy, dx)
        uy = U(dy + 1, dx) - U(dy, dx)
        n = sp.sqrt(ux ** 2 + uy ** 2 + e2)
        return ux / n, uy / n

    px_c, py_c = flux(0, 0)
    px_w, _ = flux(0, -1)
    _, py_s = flux(-1, 0)
    rhs = sp.Float(lam) * (u.center - f.center) - ((px_c - px_w) + (py_c - py_s))
    return AutoDiffOp([Assignment(g.center, rhs)], op_name='tvgrad', boundary_handling=boundary_handling, **kw)


CONFIG_SHAPES = {
    'c1': dict(factory=readme_op, shape=(20, 30), dtype='float32'),
    'c2': dict(factory=diffusion2d_op, shape=(8192, 8192), dtype='float32'),
    'c3': dict(factory=heat3d_op, shape=(1024, 1024, 1024), dtype='float32'),
    'c4': dict(factory=stencil27_op, shape=(768, 768, 768), dtype='float64'),
    'c5': dict(factory=tv_gradient_op, shape=(16, 4096, 4096), dtype='float32'),
}


def make_config(name, shape=None, dtype=None, **kw):
    c = CONFIG_SHAPES[name]
    return c['factory'](shape=shape or c['shape'], dtype=dtype or c['dtype'], **kw)
