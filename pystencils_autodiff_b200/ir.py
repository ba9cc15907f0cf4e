"""StencilIR: the lowered form of one kernel (forward or backward) that the CUDA emitter consumes.

This replaces what the reference obtains from ``pystencils.create_kernel(assignments, ghost_layers=…,
target='gpu')`` at /root/reference/src/pystencils_autodiff/_autodiff.py:495-508,528-542: the iteration space and
the per-field access sets of one ``AssignmentCollection``.

Iteration-space rule (SURVEY.md Appendix A-3, restated from pystencils' ``create_kernel``):

* ``boundary_handling=None``  → cells ``gl <= c_k < N_k - gl`` on every axis, ``gl = max |offset|`` over all accesses
  of *this* kernel; every other cell of an output is 0 (the reference gets that from ``torch.zeros``,
  backends/_torch_native.py:64,108 — here the kernel writes the zeros itself).
* ``'zeros'`` → all cells, every offset read that falls outside the array evaluates to 0
  (transformations.py:12-36, ghost_layers=0 at _autodiff.py:499,534).
"""
from dataclasses import dataclass, field as dc_field
from typing import Dict, List, Tuple

import numpy as np
import sympy as sp

from .assignment import AssignmentCollection, coerce_assignments
from .field import BFLOAT16, Field
from .transformations import ConditionalFieldAccess

__all__ = ['StencilKernelIR', 'KernelParameter', 'lower_assignments', 'split_index_components']


@dataclass
class KernelParameter:
    """One entry of the kernel's call signature (fields first, then scalars), like the reference wrapper's
    ``call_<kernel>(at::Tensor& f…, double a…)`` parameters (backends/astnodes.py:143-146)."""
    name: str
    is_field: bool
    dtype: np.dtype
    field: object = None

    @property
    def symbol(self):
        return sp.Symbol(self.name)


@dataclass
class StencilKernelIR:
    function_name: str
    ndim: int
    boundary: str                       # 'none' | 'zeros'
    ghost_layers: int                   # interior margin for 'none'; 0 for 'zeros'
    input_fields: List[Field]
    output_fields: List[Field]
    scalars: List[sp.Symbol]
    subexpressions: List[Tuple[sp.Symbol, sp.Expr]]
    main: List[Tuple[Field.Access, sp.Expr]]
    read_accesses: Dict[str, List[Field.Access]] = dc_field(default_factory=dict)
    lhs_offset: Tuple[int, ...] = ()
    assignments: AssignmentCollection = None
    compute_dtype: np.dtype = None
    fast_math: bool = False             # opt-in: flush-to-zero, approximate division / sqrt (like pystencils' fast approximations)

    # -- reference-compatible introspection (``_backport.py:20-29``: fields_read / fields_written) -----------
    @property
    def fields_read(self):
        return set(self.input_fields)

    @property
    def fields_written(self):
        return set(self.output_fields)

    @property
    def fields_accessed(self):
        return set(self.input_fields) | set(self.output_fields)

    @property
    def all_fields(self):
        """Kernel field order: outputs (sorted) then inputs (sorted); a field that is read *and* written
        (``+=`` accumulation for time-constant fields, _autodiff.py:110-113) appears once, as an output."""
        outs = list(self.output_fields)
        return outs + [f for f in self.input_fields if f not in outs]

    def get_parameters(self):
        params = [KernelParameter(f.name, True, f.dtype.numpy_dtype, f) for f in self.all_fields]
        params += [KernelParameter(s.name, False, np.dtype(np.float64)) for s in self.scalars]
        return params

    # -- geometry ----------------------------------------------------------------------------------------------
    def halo(self, field_name) -> List[Tuple[int, int]]:
        """Per axis ``(lo, hi)`` = how far below / above the centre this field is read."""
        res = [[0, 0] for _ in range(self.ndim)]
        for a in self.read_accesses.get(field_name, []):
            for k, o in enumerate(a.offsets):
                res[k][0] = max(res[k][0], -int(o))
                res[k][1] = max(res[k][1], int(o))
        return [tuple(r) for r in res]

    @property
    def max_halo(self):
        res = [[0, 0] for _ in range(self.ndim)]
        for f in self.input_fields:
            for k, (lo, hi) in enumerate(self.halo(f.name)):
                res[k][0] = max(res[k][0], lo)
                res[k][1] = max(res[k][1], hi)
        return [tuple(r) for r in res]

    def bytes_per_cell(self):
        """Algorithmic (compulsory) HBM bytes per cell: every read field once + every written field once."""
        b = 0
        for f in self.all_fields:
            n = int(np.prod([int(s) for s in f.index_shape])) if f.index_dimensions else 1
            rw = (1 if f in self.input_fields else 0) + (1 if f in self.output_fields else 0)
            b += rw * n * f.dtype.itemsize
        return b

    def __str__(self):
        return 'StencilKernelIR(%s, ndim=%d, boundary=%s, gl=%d, in=%s, out=%s)' % (
            self.function_name, self.ndim, self.boundary, self.ghost_layers,
            [f.name for f in self.input_fields], [f.name for f in self.output_fields])


def _strip_conditional(expr):
    """Unwrap ConditionalFieldAccess nodes (value 0 when out of bounds); returns (expr, found_any)."""
    cfas = list(expr.atoms(ConditionalFieldAccess))
    if not cfas:
        return expr, False
    for c in cfas:
        if c.outofbounds_value != 0:
            raise NotImplementedError('only outofbounds_value=0 is supported')
    return expr.xreplace({c: c.access for c in cfas}), True


def lower_assignments(assignments, boundary_handling=None, function_name='kernel', ghost_layers=None,
                      data_type=None, fast_math=False) -> StencilKernelIR:
    ac = coerce_assignments(assignments)
    boundary = 'zeros' if (boundary_handling is not None and str(getattr(boundary_handling, 'value', boundary_handling)) == 'zeros') else 'none'

    subexpressions, main = [], []
    found_guard = False
    for a in ac.subexpressions:
        rhs, g = _strip_conditional(a.rhs)
        found_guard |= g
        subexpressions.append((a.lhs, rhs))
    for a in ac.main_assignments:
        if not isinstance(a.lhs, Field.Access):
            raise ValueError('main assignments must write to a field access')
        rhs, g = _strip_conditional(a.rhs)
        found_guard |= g
        main.append((a.lhs, rhs))
    if found_guard:
        boundary = 'zeros'
    if not main:
        raise ValueError('no main assignments')

    clean = AssignmentCollection({l: r for l, r in main}, {l: r for l, r in subexpressions})
    # every access on a right-hand side — including a ``+=`` form's read of its own output, which pystencils'
    # ``free_symbols`` (rhs symbols minus bound symbols) does not list
    reads = sorted(set().union(*[r.atoms(Field.Access) for _, r in subexpressions + main]), key=str)
    writes = [l for l, _ in main]
    scalars = sorted([s for s in clean.free_symbols if not isinstance(s, Field.Access)], key=str)

    all_acc = reads + writes
    ndims = {a.field.spatial_dimensions for a in all_acc}
    if len(ndims) != 1:
        raise ValueError('all fields of a kernel must have the same number of spatial dimensions')
    ndim = ndims.pop()
    if not 1 <= ndim <= 3:
        raise NotImplementedError('1, 2 or 3 spatial dimensions are supported')
    for a in all_acc:
        if not all(isinstance(o, int) for o in a.offsets):
            raise NotImplementedError('only integer (relative) offsets are supported: %s' % a)
        if a.field.index_dimensions > 1:
            raise NotImplementedError('at most one index dimension is supported')
        if a.field.index_dimensions and not a.field.has_fixed_index_shape:
            raise NotImplementedError('index shape must be fixed')

    lhs_offsets = {tuple(w.offsets) for w in writes}
    if len(lhs_offsets) != 1:
        raise NotImplementedError('all main assignments must write at the same relative offset')
    lhs_offset = lhs_offsets.pop()
    seen = set()
    for w in writes:
        key = (w.field, w.index)
        if key in seen:
            raise ValueError('kernel writes %s twice' % (w,))
        seen.add(key)

    if boundary == 'zeros':
        if any(o != 0 for o in lhs_offset):
            raise NotImplementedError("'zeros' boundary handling needs centre writes")
        gl = 0
    elif ghost_layers is not None:
        gl = int(ghost_layers)
    else:
        gl = max([a.required_ghost_layers for a in all_acc] + [0])

    read_accesses: Dict[str, List[Field.Access]] = {}
    for a in reads:
        read_accesses.setdefault(a.field.name, []).append(a)
    input_fields = sorted({a.field for a in reads}, key=str)
    output_fields = sorted({a.field for a in writes}, key=str)
    names = [f.name for f in set(input_fields) | set(output_fields)]
    if len(names) != len(set(names)):
        raise ValueError('two different fields share a name: %s' % sorted(names))

    if data_type is not None:
        cdt = np.dtype({'double': np.float64, 'float': np.float32}.get(data_type, data_type))
    else:
        # bfloat16 computes in fp32 at least: np.result_type cannot promote the stand-in dtype
        cdt = np.result_type(*[np.float32 if f.dtype.numpy_dtype == BFLOAT16 else f.dtype.numpy_dtype
                               for f in input_fields + output_fields])
        if cdt.kind != 'f':
            cdt = np.dtype(np.float64)
        if cdt.itemsize < 4:
            cdt = np.dtype(np.float32)

    return StencilKernelIR(function_name=function_name, ndim=ndim, boundary=boundary, ghost_layers=gl,
                           input_fields=input_fields, output_fields=output_fields, scalars=scalars,
                           subexpressions=subexpressions, main=main, read_accesses=read_accesses,
                           lhs_offset=lhs_offset, assignments=clean, compute_dtype=cdt, fast_math=bool(fast_math))


def split_index_components(ir: StencilKernelIR):
    """Rewrite a kernel over fields with one index dimension as a kernel over scalar *component fields*.

    ``v[offsets](i)`` becomes ``v__i[offsets]``: with a structure-of-arrays layout (x contiguous — the ``fzyx`` layout
    the reference's lattice-Boltzmann code uses on GPUs, lbm/_autodiff_lbstep.py:69-86) component ``i`` of ``v`` is an
    ordinary scalar field starting ``i * stride_index`` elements after ``v``, so the fast kernels apply unchanged.
    Returns ``(scalar_ir, components)`` with ``components[name__i] = (original field name, i)``, or ``(ir, {})`` when no
    field has an index dimension."""
    if not any(f.index_dimensions for f in ir.all_fields):
        return ir, {}
    components, repl, cache = {}, {}, {}

    def comp_field(f, i):
        key = (f.name, i)
        if key not in cache:
            nf = Field.create_fixed_size('%s__%d' % (f.name, i), tuple(f.spatial_shape), 0, f.dtype.numpy_dtype) \
                if f.has_fixed_shape else Field.create_generic('%s__%d' % (f.name, i), f.spatial_dimensions,
                                                               f.dtype.numpy_dtype)
            cache[key] = nf
            components[nf.name] = (f.name, i)
        return cache[key]

    def conv(a):
        if not a.field.index_dimensions:
            return a
        return Field.Access(comp_field(a.field, int(a.index[0])), a.offsets)

    accesses = set()
    for _, r in ir.subexpressions + ir.main:
        accesses |= r.atoms(Field.Access)
    for a in accesses:
        repl[a] = conv(a)
    sub = {l: r.xreplace(repl) for l, r in ir.subexpressions}
    main = {conv(l): r.xreplace(repl) for l, r in ir.main}
    scalar_ir = lower_assignments(AssignmentCollection(main, sub), 'zeros' if ir.boundary == 'zeros' else None,
                                  ir.function_name, ghost_layers=ir.ghost_layers if ir.boundary != 'zeros' else None,
                                  data_type=ir.compute_dtype, fast_math=ir.fast_math)
    return scalar_ir, components


def lift_to_3d(ir: StencilKernelIR):
    """A 2-D kernel as a 3-D kernel over fields with a leading extent-1 dimension (offset 0 along it): the tensor
    ``t[Y, X]`` is passed as ``t[None]``.  Lets 2-D stencils use machinery that exists for the 3-D march only (the
    fused-step kernels).  Only for ``'zeros'`` boundary handling: an inferred ghost width would also apply to the new
    dimension and leave nothing to iterate."""
    if ir.ndim != 2:
        raise ValueError('lift_to_3d expects a 2-D kernel')
    if ir.boundary != 'zeros':
        raise ValueError("lift_to_3d needs boundary_handling='zeros'")
    if any(f.index_dimensions for f in ir.all_fields):
        raise ValueError('lift_to_3d expects scalar fields')
    cache = {}

    def lifted(f):
        if f.name not in cache:
            cache[f.name] = Field.create_fixed_size(f.name, (1,) + tuple(f.spatial_shape), 0, f.dtype.numpy_dtype) \
                if f.has_fixed_shape else Field.create_generic(f.name, 3, f.dtype.numpy_dtype)
        return cache[f.name]

    def conv(a):
        return Field.Access(lifted(a.field), (0,) + tuple(a.offsets))

    accesses = set()
    for _, r in ir.subexpressions + ir.main:
        accesses |= r.atoms(Field.Access)
    repl = {a: conv(a) for a in accesses}
    sub = {l: r.xreplace(repl) for l, r in ir.subexpressions}
    main = {conv(l): r.xreplace(repl) for l, r in ir.main}
    return lower_assignments(AssignmentCollection(main, sub), 'zeros', ir.function_name, data_type=ir.compute_dtype,
                             fast_math=ir.fast_math)
