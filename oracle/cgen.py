"""CPU oracle — "restated pystencils CPU path": C/OpenMP loop nests for stencil assignments.
TEST / BASELINE INFRASTRUCTURE, NOT PRODUCT CODE (see ``oracle/evaluate.py`` for the rules and parity status:
*parity unpinned* — pystencils itself is unavailable, this restates what its CPU backend generates).

What is restated (SURVEY.md §8d, Appendix C; reference call sites
/root/reference/src/pystencils_autodiff/_autodiff.py:479-492,510-525,544-560 →
``pystencils.create_kernel(..., cpu_openmp=True).compile()``):

* one loop per spatial axis, outermost ``#pragma omp parallel for schedule(static)``, innermost over the
  contiguous axis, ``restrict`` pointers, int64 index arithmetic with per-field strides;
* ``boundary_handling=None`` → interior iteration with ghost width ``max |offset|``; ``'zeros'`` → full
  iteration, every offset read guarded by a ternary (transformations.py:26-30);
* arithmetic in ``double`` regardless of the field dtype (pystencils' ``data_type='double'`` default), rounded on
  store; compiled with pystencils' default cpujit flag set ``-Ofast -DNDEBUG -fPIC -march=native -fopenmp``
  (``flavour='fast'``, used for timing) or ``-O2 -ffp-contract=off`` (``flavour='strict'``, used as a checker).
"""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import sympy as sp
from sympy.printing.c import C99CodePrinter

from ._model import as_collection, field_dtype, ghost_width, is_access, offsets_of

# $PSAD_ORACLE_BUILD_DIR: compile outside the tree (bench.py uses a temporary directory: the tree may be read-only)
_BUILD_DIR = os.environ.get('PSAD_ORACLE_BUILD_DIR') or os.path.join(os.path.dirname(os.path.abspath(__file__)), '_build')
_CTYPES = {np.dtype(np.float32): 'float', np.dtype(np.float64): 'double'}

FLAGS = {
    'fast': ['-Ofast', '-DNDEBUG', '-fPIC', '-march=native', '-fopenmp', '-std=c99'],
    'strict': ['-O2', '-fPIC', '-fopenmp', '-std=c99', '-ffp-contract=off'],
}


class _Printer(C99CodePrinter):
    def _print_Pow(self, expr):
        b, e = expr.base, expr.exp
        if e.is_Integer and 1 < abs(int(e)) <= 4:
            s = '*'.join(['(%s)' % self._print(b)] * abs(int(e)))
            return s if int(e) > 0 else '(1.0/(%s))' % s
        if e == -1:
            return '(1.0/(%s))' % self._print(b)
        return super()._print_Pow(expr)


def _mode(boundary_handling):
    v = getattr(boundary_handling, 'value', boundary_handling)
    return 'none' if v is None else str(v)


def generate_c(assignments, boundary_handling=None, function_name='kernel', openmp=True):
    """Returns ``(c_source, field_names, scalar_names)``; the function signature is
    ``void f(void** fields, const int64_t* shape, const int64_t* strides, const double* scalars)`` with
    ``strides[f*4 + d]`` in elements."""
    ac = as_collection(assignments)
    mode = _mode(boundary_handling)
    reads = ac.reads()
    writes = [a.lhs for a in ac.main_assignments]
    scalars = sorted([s for s in ac.free_symbols if not is_access(s)], key=str)
    out_fields = sorted({w.field for w in writes}, key=str)
    in_fields = sorted({r.field for r in reads}, key=str)
    all_fields = out_fields + [f for f in in_fields if f not in out_fields]
    fidx = {f.name: i for i, f in enumerate(all_fields)}
    ndim = all_fields[0].spatial_dimensions
    gl = 0 if mode == 'zeros' else max([ghost_width(a) for a in reads + writes] + [0])

    pr = _Printer()
    lines = ['#include <stdint.h>', '#include <math.h>', '',
             'void %s(void** fields, const int64_t* shape, const int64_t* strides, const double* scalars)' % function_name,
             '{']
    for f in all_fields:
        ct = _CTYPES[field_dtype(f)]
        const = '' if f in out_fields else 'const '
        lines.append('  %s%s* restrict _data_%s = (%s%s*) fields[%d];' % (const, ct, f.name, const, ct, fidx[f.name]))
    for k in range(ndim):
        lines.append('  const int64_t _size_%d = shape[%d];' % (k, k))
    for f in all_fields:
        for k in range(ndim + f.index_dimensions):
            lines.append('  const int64_t _stride_%s_%d = strides[%d];' % (f.name, k, fidx[f.name] * 4 + k))
    for i, s in enumerate(scalars):
        lines.append('  const double %s = scalars[%d];' % (s.name, i))

    def addr(a):
        terms = ['_stride_%s_%d*(ctr_%d%+d)' % (a.field.name, k, k, int(o)) for k, o in enumerate(offsets_of(a))]
        terms += ['_stride_%s_%d*%d' % (a.field.name, ndim + j, int(i)) for j, i in enumerate(a.index)]
        return '_data_%s[%s]' % (a.field.name, ' + '.join(terms))

    def read_expr(a):
        if mode == 'zeros' and any(o != 0 for o in offsets_of(a)):
            conds = []
            for k, o in enumerate(offsets_of(a)):
                if o != 0:
                    conds.append('ctr_%d%+d < 0 || ctr_%d%+d >= _size_%d' % (k, int(o), k, int(o), k))
            return '((%s) ? 0.0 : (double) %s)' % (' || '.join(conds), addr(a))
        return '(double) %s' % addr(a)

    for k in range(ndim):
        ind = '  ' * (k + 1)
        if k == 0 and openmp:
            lines.append(ind + '#pragma omp parallel for schedule(static)')
        lines.append(ind + 'for (int64_t ctr_%d = %d; ctr_%d < _size_%d - %d; ++ctr_%d)' % (k, gl, k, k, gl, k))
        lines.append(ind + '{')
    ind = '  ' * (ndim + 1)
    local = {}
    for i, a in enumerate(reads):
        name = '_r%d' % i
        local[a] = sp.Symbol(name)
        lines.append(ind + 'const double %s = %s;' % (name, read_expr(a)))
    for a in ac.subexpressions:
        lines.append(ind + 'const double %s = %s;' % (pr.doprint(a.lhs), pr.doprint(a.rhs.xreplace(local))))
    for a in ac.main_assignments:
        ct = _CTYPES[field_dtype(a.lhs.field)]
        lines.append(ind + '%s = (%s) (%s);' % (addr(a.lhs), ct, pr.doprint(a.rhs.xreplace(local))))
    for k in reversed(range(ndim)):
        lines.append('  ' * (k + 1) + '}')
    lines.append('}')
    return '\n'.join(lines) + '\n', [f.name for f in all_fields], [s.name for s in scalars]


class CompiledCKernel:
    """ctypes handle on a compiled loop nest; call with numpy arrays as keyword arguments (like a pystencils
    kernel: ``kernel(x=x, y=y, z=z, a=5.)``, tests/backends/test_torch_native_compilation.py:183)."""

    def __init__(self, lib_path, function_name, field_names, scalar_names, source, fields):
        self.lib = ctypes.CDLL(lib_path)
        self.fn = getattr(self.lib, function_name)
        self.fn.restype = None
        self.field_names = field_names
        self.scalar_names = scalar_names
        self.code = source
        self._fields = {f.name: f for f in fields}

    def __call__(self, **kwargs):
        arrs = [kwargs[n] for n in self.field_names]
        ndim = self._fields[self.field_names[0]].spatial_dimensions
        shape = (ctypes.c_int64 * 3)(*([int(s) for s in arrs[0].shape[:ndim]] + [1] * (3 - ndim)))
        ptrs = (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        strides = (ctypes.c_int64 * (4 * len(arrs)))()
        for i, a in enumerate(arrs):
            assert a.dtype == field_dtype(self._fields[self.field_names[i]]), self.field_names[i]
            for d, s in enumerate(a.strides):
                strides[4 * i + d] = s // a.itemsize
        sc = (ctypes.c_double * max(1, len(self.scalar_names)))(*[float(kwargs[n]) for n in self.scalar_names])
        self.fn(ptrs, shape, strides, sc)


def _cpu_tag():
    try:
        with open('/proc/cpuinfo') as fh:
            for line in fh:
                if line.startswith('flags'):
                    return hashlib.md5(line.encode()).hexdigest()[:8]
    except OSError:
        pass
    return 'generic'


def compile_c(assignments, boundary_handling=None, function_name='kernel', flavour='fast', openmp=True):
    ac = as_collection(assignments)
    src, field_names, scalar_names = generate_c(ac, boundary_handling, function_name, openmp)
    flags = FLAGS[flavour]
    key = hashlib.md5((src + ' '.join(flags) + (_cpu_tag() if '-march=native' in flags else '')).encode()).hexdigest()
    os.makedirs(_BUILD_DIR, exist_ok=True)
    c_path = os.path.join(_BUILD_DIR, '%s_%s.c' % (function_name, key))
    so_path = os.path.join(_BUILD_DIR, '%s_%s.so' % (function_name, key))
    if not os.path.exists(so_path):
        with open(c_path, 'w') as fh:
            fh.write(src)
        tmp = so_path + '.tmp%d' % os.getpid()
        subprocess.check_call(['gcc'] + flags + ['-shared', '-o', tmp, c_path, '-lm'])
        os.replace(tmp, so_path)
    reads = set(ac.reads())
    fields = {a.field for a in reads} | {a.lhs.field for a in ac.main_assignments}
    return CompiledCKernel(so_path, function_name, field_names, scalar_names, src, fields)
