"""CUDA source emitter: instantiates the hand-written sm_100a kernel templates for one stencil.

This is the replacement of the reference's backend printer
(/root/reference/src/pystencils_autodiff/framework_integration/printer.py:12-176 together with pystencils'
``generate_c``): instead of printing a one-thread-per-cell kernel it emits a small translation unit that

* ``march`` variant — configures ``csrc/kernels/psad_march.cuh`` (persistent CTAs, TMA-staged haloed tiles in a
  shared-memory ring, mbarrier pipeline) and generates the per-step body ``psad_step``: a register window along the
  march axis (each staged element is read from shared memory once and carried in registers while its plane moves
  through the stencil), 128-bit shared loads, warp-shuffle x-halos and 128-bit streaming stores;
* ``generic`` variant — a grid-stride kernel with scalar loads for anything the fast path cannot take (unaligned
  row pitch such as the README's 20x30 fp32 fields, 1-D fields, index dimensions, off-centre writes).

Both are compiled by NVRTC for sm_100a through the C ABI (``include/psad.h``).
"""
import hashlib
import os
from dataclasses import dataclass, field as dc_field
from typing import Dict, List, Optional

import numpy as np
import sympy as sp
from sympy.codegen.ast import float32, float64, real
from sympy.printing.c import C99CodePrinter

from .field import Field
from .ir import StencilKernelIR
from .linopt import plan_linear

KERNEL_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'csrc', 'kernels')
EMITTER_VERSION = '19'

_CT = {np.dtype(np.float16): 'psad_half', np.dtype(np.float32): 'float', np.dtype(np.float64): 'double'}
_F16 = np.dtype(np.float16)
# float16 fields: storage type psad_half (psad_half.cuh), values converted to fp32 where they enter the registers
HALF_HEADER = 'psad_half.cuh'
# headers that only some kernels include: hashed into the cache key of those kernels only
_OPTIONAL_HEADERS = (HALF_HEADER,)
# AutoDiffOp(..., fast_math=True): denormals flushed, approximate reciprocal / square root (2 ulp); the explicit FMA
# chains stay as they are
FAST_MATH_OPTIONS = ['-ftz=true', '-prec-div=false', '-prec-sqrt=false']


@dataclass
class EmittedKernel:
    name: str
    kind: str                      # 'generic' | 'march'
    source: str
    ir: StencilKernelIR
    fields: List[Field]            # plan order: outputs then inputs
    scalars: List[str]
    plan: Dict = dc_field(default_factory=dict)
    # PSAD_NVRTC_EXTRA: additional compiler options for experiments (part of the cache key like every option)
    options: List[str] = dc_field(default_factory=lambda: ['-fmad=false'] + os.environ.get('PSAD_NVRTC_EXTRA', '').split())

    @property
    def cache_key(self):
        h = hashlib.md5()
        h.update(EMITTER_VERSION.encode())
        h.update(self.source.encode())
        h.update(' '.join(self.options).encode())
        for fn in sorted(os.listdir(KERNEL_DIR)):
            if fn in _OPTIONAL_HEADERS and ('#include "%s"' % fn) not in self.source:
                continue
            with open(os.path.join(KERNEL_DIR, fn), 'rb') as fh:
                h.update(fh.read())
        return '%s_%s' % (self.name[:40], h.hexdigest())


# ---------------------------------------------------------------------------------------------------------------
class _CudaPrinter(C99CodePrinter):
    """sympy -> CUDA C expression in the kernel's compute type (float literals get an ``F`` suffix)."""

    def __init__(self, compute_dtype):
        alias = {real: float32 if np.dtype(compute_dtype) == np.float32 else float64}
        super().__init__(settings={'type_aliases': alias})
        self._one = '1.0F' if np.dtype(compute_dtype) == np.float32 else '1.0'
        self._sqrt = 'sqrtf' if np.dtype(compute_dtype) == np.float32 else 'sqrt'
        self.symmap = {}   # symbol -> C text; the *expression* (and so the order of every sum) stays in terms of the
        #                    original access symbols, whatever register / variable they are mapped to

    def _print_Symbol(self, expr):
        if expr in self.symmap:
            return self.symmap[expr]
        return super()._print_Symbol(expr)

    def print_with(self, expr, symmap):
        self.symmap = symmap
        try:
            return self.doprint(expr)
        finally:
            self.symmap = {}

    # Sums are printed as explicit fused-multiply-add chains and the kernels are compiled with -fmad=false, so the
    # rounding of every cell is fixed by this printer and not by the compiler's per-instance contraction choices
    # (the step body is instantiated once per window phase; all instances must agree bit for bit, and so must
    # sharded and unsharded runs).  Long sums are split into independent accumulators to give the FMA pipes ILP.
    def _print_Add(self, expr, order=None):
        terms = list(sp.Add.make_args(expr))
        if len(terms) < 2:
            return super()._print_Add(expr, order=order)
        terms.sort(key=lambda t_: sp.default_sort_key(t_))
        n_acc = 1 if len(terms) <= 4 else (2 if len(terms) <= 9 else 4)
        chains = [terms[i::n_acc] for i in range(n_acc)]
        parts = [self._fma_chain(ch) for ch in chains if ch]
        while len(parts) > 1:
            parts = ['(%s + %s)' % (parts[i], parts[i + 1]) if i + 1 < len(parts) else parts[i]
                     for i in range(0, len(parts), 2)]
        return parts[0]

    def _fma_chain(self, terms):
        fma = 'fmaf' if self._one.endswith('F') else 'fma'
        acc = None
        for t_ in terms:
            c, rest = t_.as_coeff_Mul()
            if acc is None:
                acc = self._print(t_)
                if t_.is_Add:
                    acc = '(%s)' % acc
                continue
            if rest == 1:
                acc = '(%s + %s)' % (acc, self._print(c))
            elif c == 1 and not rest.is_Mul:
                acc = '(%s + %s)' % (acc, self._paren(rest))
            elif c == -1 and not rest.is_Mul:
                acc = '(%s - %s)' % (acc, self._paren(rest))
            else:
                if c != 1:
                    a, b = c, rest
                else:
                    a, b = rest.args[0], sp.Mul(*rest.args[1:])
                acc = '%s(%s, %s, %s)' % (fma, self._print(a), self._print(b), acc)
        return acc

    def _print_Mul(self, expr):
        # keep half-integer negative powers as *factors* (they print as psad_rsqrt(...), see _print_Pow) instead of
        # letting the stock printer turn a*b**(-1/2) into a/sqrt(b): an IEEE division plus an IEEE square root
        c, factors = expr.as_coeff_mul()
        num, den = [], []
        for f in factors:
            if f.is_Pow and f.exp.is_Rational and f.exp.is_negative and f.exp.q != 2:
                den.append(sp.Pow(f.base, -f.exp))
            else:
                num.append(f)
        if not any(f.is_Pow and f.exp.is_Rational and f.exp.q == 2 and f.exp.is_negative for f in num):
            return super()._print_Mul(expr)

        def fac(f):
            s_ = self._print(f)
            return '(%s)' % s_ if f.is_Add else s_
        parts = [fac(f) for f in num]
        if c != 1 and c != -1:
            parts.insert(0, self._print(c))
        text = '*'.join(parts)
        if den:
            text = '%s/(%s)' % (text, '*'.join(fac(f) for f in den))
        return '-(%s)' % text if c == -1 else text

    def _paren(self, e):
        s_ = self._print(e)
        return '(%s)' % s_ if (e.is_Add or e.is_Mul) else s_

    def _print_Pow(self, expr):
        b, e = expr.base, expr.exp
        if e.is_Integer and 1 < abs(int(e)) <= 8:
            base = self._print(b)
            if not (b.is_Symbol or b.is_Number):
                base = '(%s)' % base
            s = '*'.join([base] * abs(int(e)))
            return '(%s)' % s if int(e) > 0 else '(%s/(%s))' % (self._one, s)
        if e == -1:
            return '(%s/(%s))' % (self._one, self._print(b))
        if e.is_Rational and e.q == 2 and abs(int(e.p)) <= 9:
            # half-integer powers through sqrt / psad_rsqrt (<= 2 ulp) instead of pow(): x**(3/2) = x*sqrt(x),
            # x**(-3/2) = rsqrt(x)**3.  The backward of anything containing 1/sqrt(...) is full of these.
            n = int(e.p)
            if n > 0:
                root = '%s(%s)' % (self._sqrt, self._print(b))
                return root if n == 1 else '(%s*%s)' % (root, self._print(sp.Pow(b, (n - 1) // 2)))
            r = 'psad_rsqrt(%s)' % self._print(b)
            return r if n == -1 else 'psad_ipow<%d>(%s)' % (-n, r)
        return super()._print_Pow(expr)


def _c_ident(name):
    out = ''.join(ch if (ch.isalnum() or ch == '_') else '_' for ch in name)
    if not out or out[0].isdigit():
        out = '_' + out
    return out


def _is_nonlinear(ir):
    """Does any right-hand side combine field values other than by a weighted sum?  (Those kernels have expensive
    per-position terms — norms, roots, fluxes — that neighbouring cells share.)"""
    if ir.subexpressions:
        return True
    for _, rhs in ir.main:
        for node in sp.preorder_traversal(rhs):
            if isinstance(node, (sp.Pow, sp.Function)) and node.has(Field.Access):
                return True
            if isinstance(node, sp.Mul) and sum(1 for a in node.args if a.has(Field.Access)) > 1:
                return True
    return False


def _even_power_canonical(expr):
    """``(b - a)**2 -> (a - b)**2``: one sign convention under even powers, so that the same squared difference reached
    from two neighbouring cells is the same expression (bitwise the same value)."""
    def fix(pw):
        base, e = pw.args
        if e.is_Integer and e % 2 == 0 and base.could_extract_minus_sign():
            return sp.Pow(-base, e)
        return pw
    return expr.replace(lambda z: z.is_Pow, fix)


def _off3(offsets):
    return (0,) * (3 - len(offsets)) + tuple(int(o) for o in offsets)


def _kernel_name(ir, kind):
    return _c_ident('psad_%s_%s' % (ir.function_name, kind))


def _header(ir, kind, extra=''):
    lines = ['// Specialised by pystencils_autodiff_b200.emit for kernel "%s" (%s variant).' % (ir.function_name, kind),
             '// boundary=%s ghost_layers=%d ndim=%d compute=%s' % (ir.boundary, ir.ghost_layers, ir.ndim,
                                                                   _CT[ir.compute_dtype])]
    for lhs, rhs in ir.subexpressions:
        lines.append('//   %s <- %s' % (lhs, rhs))
    for lhs, rhs in ir.main:
        lines.append('//   %s <- %s' % (lhs.field_str(), rhs))
    if extra:
        lines.append(extra)
    return lines


# ---------------------------------------------------------------------------------------------------------------
def emit_generic(ir: StencilKernelIR, threads=256) -> EmittedKernel:
    name = _kernel_name(ir, 'generic')
    CT = _CT[ir.compute_dtype]
    pr = _CudaPrinter(ir.compute_dtype)
    fields = ir.all_fields
    fidx = {f.name: i for i, f in enumerate(fields)}
    scalars = [s.name for s in ir.scalars]
    lz, ly, lx = _off3(ir.lhs_offset)

    L = _header(ir, 'generic')
    L += ['#include "psad_common.cuh"']
    if any(f.dtype.numpy_dtype == _F16 for f in fields):
        L.append('#include "%s"' % HALF_HEADER)
    L += ['', 'typedef %s CT;' % CT]
    for f in fields:
        L.append('typedef %s T_%d;  // %s' % (_CT[f.dtype.numpy_dtype], fidx[f.name], f.name))
    L += ['',
          'extern "C" __global__ void __launch_bounds__(%d) %s(const __grid_constant__ PsadArgs A)' % (threads, name),
          '{',
          '  // x from the thread index (coalesced), y and z from the block indices with grid-stride loops: no 64-bit',
          '  // division per cell; pointer arithmetic is the only 64-bit work',
          '  const int nx = (int)(A.wr_hi[2] - A.wr_lo[2]), ny = (int)(A.wr_hi[1] - A.wr_lo[1]), nz = (int)(A.wr_hi[0] - A.wr_lo[0]);']
    for i, s in enumerate(scalars):
        L.append('  const CT %s = (CT)A.scalar[%d];' % (_c_ident(s), i))
    L += ['  for (int iz = blockIdx.z; iz < nz; iz += gridDim.z)',
          '  for (int iy = blockIdx.y; iy < ny; iy += gridDim.y)',
          '  for (int ix = blockIdx.x * blockDim.x + threadIdx.x; ix < nx; ix += gridDim.x * blockDim.x) {',
          '    const long long x = A.wr_lo[2] + ix;',
          '    const long long y = A.wr_lo[1] + iy;',
          '    const long long z = A.wr_lo[0] + iz;',
          '    const long long cz = z - (%d), cy = y - (%d), cx = x - (%d);  // cell the expression is evaluated at' % (lz, ly, lx),
          '    const bool inside = cz >= A.it_lo[0] && cz < A.it_hi[0] && cy >= A.it_lo[1] && cy < A.it_hi[1] &&',
          '                        cx >= A.it_lo[2] && cx < A.it_hi[2];']
    outs = []
    for k, (lhs, _) in enumerate(ir.main):
        L.append('    CT o_%d = (CT)0;' % k)
        outs.append(lhs)
    L.append('    if (inside) {')
    local = {}
    n = 0
    pre = []   # loop-invariant element offsets of every access, hoisted in front of the loops
    for fname in sorted(ir.read_accesses):
        fi = fidx[fname]
        for a in ir.read_accesses[fname]:
            dz, dy, dx = _off3(a.offsets)
            idx = int(a.index[0]) if a.index else 0
            var = 'r_%d' % n
            pre.append('  const long long off_%d = (%d) * A.stride[%d][0] + (%d) * A.stride[%d][1] + (%d) * A.stride[%d][2] + %d * A.stride[%d][3];'
                       % (n, dz, fi, dy, fi, dx, fi, idx, fi))
            addr = '((const T_%d*)A.ptr[%d])[base_%d + off_%d]' % (fi, fi, fi, n)
            n += 1
            if ir.boundary == 'zeros' and (dz or dy or dx):
                conds = []
                for o, c, d in ((dz, 'cz', 0), (dy, 'cy', 1), (dx, 'cx', 2)):
                    if o < 0:
                        conds.append('%s + (%d) >= 0' % (c, o))
                    elif o > 0:
                        conds.append('%s + (%d) < A.shape[%d]' % (c, o, d))
                L.append('      const CT %s = (%s) ? (CT)%s : (CT)0;' % (var, ' && '.join(conds), addr))
            else:
                L.append('      const CT %s = (CT)%s;' % (var, addr))
            local[a] = var
    # base offset of the evaluated cell per read field (one 64-bit multiply-add chain per field, not per access)
    base_lines = ['    const long long base_%d = cz * A.stride[%d][0] + cy * A.stride[%d][1] + cx * A.stride[%d][2];'
                  % (fidx[fname], fidx[fname], fidx[fname], fidx[fname]) for fname in sorted(ir.read_accesses)]
    at = L.index('    if (inside) {')
    L[at:at] = base_lines
    first_loop = next(i_ for i_, ln in enumerate(L) if ln.startswith('  for (int iz'))
    L[first_loop:first_loop] = pre
    for s in ir.scalars:
        local[s] = _c_ident(s.name)
    for lhs, rhs in ir.subexpressions:
        L.append('      const CT %s = %s;' % (_c_ident(lhs.name), pr.print_with(rhs, local)))
        local[lhs] = _c_ident(lhs.name)
    for k, (lhs, rhs) in enumerate(ir.main):
        L.append('      o_%d = %s;' % (k, pr.print_with(rhs, local)))
    L.append('    }')
    for k, lhs in enumerate(outs):
        fi = fidx[lhs.field.name]
        idx = int(lhs.index[0]) if lhs.index else 0
        L.append('    ((T_%d*)A.ptr[%d])[z * A.stride[%d][0] + y * A.stride[%d][1] + x * A.stride[%d][2] + %d * A.stride[%d][3]] = (T_%d)o_%d;'
                 % (fi, fi, fi, fi, fi, idx, fi, fi, k))
    L += ['  }', '}', '']

    plan = dict(kind=0, ndim=ir.ndim, n_fields=len(fields), n_scalars=len(scalars), threads=threads, smem_bytes=0,
                tile_x=0, tile_y=0, chunk=0, ctas_per_sm=8, boundary=1 if ir.boundary == 'zeros' else 0,
                ghost_layers=ir.ghost_layers,
                fields=[dict(elem_size=f.dtype.itemsize, is_input=int(f in ir.input_fields),
                             is_output=int(f in ir.output_fields),
                             index_size=int(f.index_shape[0]) if f.index_dimensions else 1, tma=0, box=(0, 0, 0))
                        for f in fields])
    ek = EmittedKernel(name, 'generic', '\n'.join(L), ir, fields, scalars, plan)
    if ir.fast_math:
        ek.options = ek.options + FAST_MATH_OPTIONS
    return ek


# ---------------------------------------------------------------------------------------------------------------
@dataclass
class MarchTuning:
    """Tile geometry of the march template.  ``sx`` cells per thread along x (one warp spans a tile row, so the
    tile is 32*sx cells wide), ``ry`` rows per thread, ``ty`` rows per tile, ``stages`` ring slots,
    ``chunk`` planes (3-D) / row tiles (2-D) per work item (0 = whole axis, balanced by the runtime)."""
    sx: int = 0
    ry: int = 0
    ty: int = 0
    lookahead: int = 0     # staged planes in flight ahead of the consumers (0 = measured optimum: 3 for fp32, 4 for fp64)
    stages: int = 0        # ring slots (0 = slots still being read + lookahead)
    chunk: int = 0
    min_ctas: int = 0
    ctas_per_sm: int = 0   # cap on resident CTAs per SM (0 = whatever fits)
    carry: bool = True     # keep staged elements in registers while their plane moves through the stencil
    plane_sums: bool = True  # 3-D: evaluate in-plane sub-sums shared by several z-offsets once per plane and carry them
    linopt: bool = True      # shared partial sums across the cells of a thread for linear plane sums (linopt.py)
    arrival: Optional[bool] = None  # evaluate EVERY per-plane group of the sum when its plane arrives and carry only
    #                                 scalars (no raw values); default: when the stencil has more than 9 accesses
    cross_cse: Optional[bool] = None   # common subexpressions across ALL cells of a thread (default: non-linear
    #                                    stencils, whose neighbouring cells share fluxes / norms / reciprocal roots)
    exchange: Optional[bool] = None    # fused-step kernels (emit_chain.py): pass intermediate rows between warps through
    #                                    shared memory (one consumer barrier per plane) instead of recomputing them
    store_mode: int = 1    # global store cache policy: 0 default, 1 streaming (.cs, default), 2 write-through
    shuffle: Optional[bool] = None   # x-halo elements from neighbouring lanes instead of shared memory
    #                                  (default: yes; scalar LDS halos only win for narrow fp64 strips)
    lds_pair: Optional[bool] = None  # 8-byte fields, 4-cell strips: fetch a lane's two 16-byte vectors in an order that
    #                                  depends on the lane, so that no LDS.128 has a bank conflict (psad_lds_pair).  Default
    #                                  OFF: measured on B200 (profiles/r2_c4_bank_conflicts.md) the 40 extra selects per
    #                                  step cost more than the conflicts (27-point fp64: 1.13 -> 1.30 ms at full clocks)


def march_ineligible_reason(ir: StencilKernelIR) -> Optional[str]:
    if ir.ndim not in (2, 3):
        return 'needs 2 or 3 spatial dimensions'
    if any(o != 0 for o in ir.lhs_offset):
        return 'off-centre writes'
    for f in ir.all_fields:
        if f.index_dimensions:
            return 'index dimensions'
        if f.dtype.numpy_dtype not in (_F16, np.dtype(np.float32), np.dtype(np.float64)):
            return 'only float16/float32/float64 fields'
    if len({f.dtype.numpy_dtype for f in ir.all_fields}) > 1 and any(f.dtype.numpy_dtype == _F16 for f in ir.all_fields):
        return 'float16 fields mixed with wider fields'
    if not ir.input_fields:
        return 'no input fields'
    for f in ir.input_fields:
        if f in ir.output_fields and any(any(o != 0 for o in a.offsets) for a in ir.read_accesses[f.name]):
            return 'in-place update of a field read at an offset'
    if len(ir.all_fields) > 12:
        return 'too many fields'
    return None


def emit_march(ir: StencilKernelIR, tuning: Optional[MarchTuning] = None, masked: bool = True, peer: bool = False) -> EmittedKernel:
    """Emit the march variant; when the default tile does not fit (several wide-halo fp64 fields), fall back to
    shallower prefetch and then to smaller tiles — unless the caller pinned those parameters.

    ``peer``: the peer-halo instance (3-D only) — ghost planes along dim 0 are staged by TMA straight from the neighbouring
    GPUs' arrays (``psad_kernel_launch_peer``, ``PSAD_PEER`` in psad_march.cuh); the per-step body is the same."""
    import dataclasses
    t = tuning or MarchTuning()
    candidates = [t]
    if not t.lookahead and not t.stages:
        candidates += [dataclasses.replace(t, lookahead=la) for la in (3, 2)]
    if not t.ty and not t.ry:
        for ry, ty in ((2, 30), (2, 14), (1, 15), (1, 7)):
            candidates += [dataclasses.replace(t, ry=ry, ty=ty, lookahead=t.lookahead or (2 if ty < 30 else 0))]
    last = None
    for cand in candidates:
        try:
            return _emit_march(ir, cand, masked, peer)
        except ValueError as e:
            last = e
            if 'shared memory' not in str(e) and 'threads' not in str(e):
                raise
    raise last


def _emit_march(ir: StencilKernelIR, tuning: Optional[MarchTuning] = None, masked: bool = True, peer: bool = False) -> EmittedKernel:
    reason = march_ineligible_reason(ir)
    if reason:
        raise ValueError('march variant not applicable: ' + reason)
    if peer and ir.ndim != 3:
        raise ValueError('march variant not applicable: peer halos need 3-D fields')
    t = tuning or MarchTuning()
    if t.shuffle is None:
        import dataclasses
        t = dataclasses.replace(t, shuffle=True)
    # masked=False: every written cell is inside the iteration range ('zeros' boundary, or a launch range whose
    # iteration and write parts coincide) -> no per-cell select, no mask bookkeeping
    name = _kernel_name(ir, ('march' if masked else 'march_nomask') + ('_peer' if peer else ''))
    CT = _CT[ir.compute_dtype]
    pr = _CudaPrinter(ir.compute_dtype)
    fields = ir.all_fields
    fidx = {f.name: i for i, f in enumerate(fields)}
    scalars = [s.name for s in ir.scalars]
    nd = ir.ndim
    max_esize = max(f.dtype.itemsize for f in fields)
    half = max_esize == 2     # all fields float16 (march_ineligible_reason): 8-byte vectors of 4 halves, fp32 window

    def vec_cells(es):       # cells per shared load / global store vector
        return 4 if es == 2 else 16 // es

    def reg_type(f):         # type of an output field's results in registers (rounded to fp16 only by the store)
        return CT if f.dtype.itemsize == 2 else _CT[f.dtype.numpy_dtype]

    # ---- geometry ------------------------------------------------------------------------------------------
    SX = t.sx or 4   # cells per thread along x: one 16-byte vector for 4-byte types, two for 8-byte types, one 8-byte
    #                  vector for float16 (8 halves per lane would make the box 256 + pads wide: over the TMA limit)
    if half and SX % 4:
        raise ValueError('sx must be a multiple of 4 for float16 fields')
    if not half and (SX * min(f.dtype.itemsize for f in fields)) % 16:
        raise ValueError('sx*itemsize must be a multiple of 16 bytes')
    TX = 32 * SX
    mh = ir.max_halo                        # per ndim axis (lo, hi)
    mh3 = [(0, 0)] * (3 - nd) + list(mh)
    HZL, HZH = (mh3[0] if nd == 3 else (0, 0))
    D = HZL + HZH
    # measured on B200 (scripts/sweep.py, profiles/): fp32 3-D 32x128 tiles / 2 rows per thread, fp32 2-D 16x128 / 1 row,
    # fp64 21x128 tiles / 3 rows, x-halos by warp shuffle (27-pt: 6.44 TB/s)
    cross_cse = _is_nonlinear(ir) if t.cross_cse is None else bool(t.cross_cse)
    if max_esize <= 4:
        RY = t.ry or (2 if nd == 3 else 1)
        # cross-cell CSE keeps the shared temporaries of all the thread's cells live: 15+1 warps (128 registers) instead
        # of 16+1 (96) — TV-gradient adjoint 0.758 -> 0.722 ms, and 1.00 ms when it has to spill
        # float16: the conversions take the 15+1-warp CSE tile over 128 registers (36 bytes spilled); 11+1 warps fit
        TY = t.ty or (((22 if half else 30) if cross_cse else 32) if nd == 3 else 16)
    else:
        # 7 consumer warps + the producer warp = 8 warps: ptxas budgets registers for the CTA size rounded up to 4
        # warps, so 8+1 warps would be capped at 168 registers and spill (the 27-point window needs ~240)
        RY = t.ry or 3
        TY = t.ty or 7 * RY
    if TY % RY:
        raise ValueError('ty must be a multiple of ry')
    THREADS = 32 * (TY // RY)
    if THREADS + 32 > 1024:
        raise ValueError('tile too tall: %d threads' % THREADS)

    tma_fields = [f for f in fields if f in ir.input_fields]   # plan order: the runtime numbers tensor maps this way
    geo = {}
    off = 0
    for ti, f in enumerate(tma_fields):
        h3 = [(0, 0)] * (3 - nd) + list(ir.halo(f.name))
        es = f.dtype.itemsize
        vec = vec_cells(es)
        pad = 16 // es       # pads in whole 16-byte units: box rows stay a multiple of 16 bytes, lane loads aligned
        hxl, hxr = h3[2]
        if hxl > SX or hxr > SX:
            raise ValueError('x halo wider than the per-thread strip')
        padl = -(-hxl // pad) * pad
        padr = -(-hxr // pad) * pad
        boxw = TX + padl + padr
        boxh = TY + h3[1][0] + h3[1][1]
        if boxw > 256 or boxh > 256:
            raise ValueError('TMA box too large')
        nbytes = boxw * boxh * es
        geo[f.name] = dict(ti=ti, es=es, vec=vec, nv=SX // vec, hz=h3[0], hy=h3[1], hx=h3[2], padl=padl, boxw=boxw,
                           boxh=boxh, bytes=nbytes, off=off, T=_CT[f.dtype.numpy_dtype],
                           Tw='float' if es == 2 else _CT[f.dtype.numpy_dtype], ww=max(1, es // 4))   # window: fp16 as float
        off += -(-nbytes // 128) * 128
    STAGE_BYTES = off
    # ---- plane partial sums --------------------------------------------------------------------------------------
    # rhs = sum_dz G_dz(accesses of plane z+dz) + rest.  Where G_a and G_b are the same expression up to the z shift
    # (e.g. the z-1 and z+1 planes of a symmetric stencil), the value Q(plane) is computed once per cell when the plane
    # enters the window at the highest of these positions and carried down in registers; the raw elements of that
    # plane are then not needed at the lower positions at all.
    q_classes = []           # [{canon: expr at dz=0, members: [dz...], hi: dz}]
    main_exprs = []          # per main assignment: expression over accesses and Q symbols
    raw_accesses = {f.name: set() for f in tma_fields}

    def _zshift(expr, dz):
        return expr.xreplace({a: a.get_shifted(*([dz] + [0] * (nd - 1))) for a in expr.atoms(Field.Access)})

    use_q = bool(t.plane_sums and t.carry and nd == 3 and D > 0 and not ir.subexpressions)
    n_reads = sum(len(v) for v in ir.read_accesses.values())
    arrival = use_q and (t.arrival if t.arrival is not None else n_reads > 9)
    for lhs, rhs in ir.main:
        rest = []
        groups = {}
        if use_q:
            for term in sp.Add.make_args(rhs):
                dzs = {int(a.offsets[0]) for a in term.atoms(Field.Access)}
                if len(dzs) == 1:
                    groups.setdefault(dzs.pop(), []).append(term)
                else:
                    rest.append(term)
        else:
            rest = [rhs]
        by_canon = {}
        for dz, terms in groups.items():
            g_expr = sp.Add(*terms)
            by_canon.setdefault(_zshift(g_expr, -dz), []).append(dz)
        new_terms = list(rest)
        for canon, members in by_canon.items():
            n_acc = len(canon.atoms(Field.Access))
            if arrival and members == [HZH]:
                new_terms += [_zshift(canon, HZH)]      # used in the step it arrives: nothing to carry
            elif (arrival and n_acc >= 1) or (len(members) >= 2 and n_acc >= 2):
                ci = None
                for i_, qc in enumerate(q_classes):
                    if qc['canon'] == canon:
                        ci = i_
                        qc['members'] = sorted(set(qc['members']) | set(members))
                if ci is None:
                    q_classes.append(dict(canon=canon, members=sorted(members)))
                    ci = len(q_classes) - 1
                new_terms += [sp.Symbol('psadQ_%d_%d' % (ci, dz + HZL)) for dz in members]
            else:
                new_terms += [_zshift(canon, dz) for dz in members]
        main_exprs.append((lhs, sp.Add(*new_terms)))
    for qc in q_classes:
        qc['hi'] = HZH if arrival else max(qc['members'])
        qc['lo'] = min(qc['members'])
        qc['expr_hi'] = _zshift(qc['canon'], qc['hi'])
    for _, e in main_exprs:
        for a in e.atoms(Field.Access):
            raw_accesses[a.field.name].add(a)
    for qc in q_classes:
        for a in qc['expr_hi'].atoms(Field.Access):
            raw_accesses[a.field.name].add(a)
    for lhs_, e in ir.subexpressions:
        for a in e.atoms(Field.Access):
            raw_accesses[a.field.name].add(a)

    # ---- register-window analysis ------------------------------------------------------------------------------
    # unit = ('U', row, v): aligned 16-byte vector v of the thread's own strip in tile row `row` (relative to the
    # thread's first row);  ('H', row, c): single halo element at strip column c (<0 or >=SX).
    def src_col(c):
        return SX + c if c < 0 else c - SX

    need = {f.name: [set() for _ in range(D + 1)] for f in tma_fields}
    for f in tma_fields:
        g = geo[f.name]
        for a in sorted(raw_accesses[f.name], key=str):
            dz, dy, dx = _off3(a.offsets)
            j = dz + HZL
            for r in range(RY):
                for c in range(SX):
                    cc = c + dx
                    if 0 <= cc < SX:
                        need[f.name][j].add(('U', r + dy, cc // g['vec']))
                    else:
                        need[f.name][j].add(('H', r + dy, cc))
                        if t.shuffle:
                            need[f.name][j].add(('U', r + dy, src_col(cc) // g['vec']))
    carried = {f.name: [set() for _ in range(D + 1)] for f in tma_fields}   # available from the previous step
    held = {f.name: [set() for _ in range(D + 1)] for f in tma_fields}
    fresh = {f.name: [set() for _ in range(D + 1)] for f in tma_fields}
    for f in tma_fields:
        nm = f.name
        for j in range(D, -1, -1):
            future = set().union(*[need[nm][jj] for jj in range(j)]) if j > 0 else set()
            if j < D and t.carry:
                carried[nm][j] = held[nm][j + 1] & (need[nm][j] | future)
            held[nm][j] = need[nm][j] | carried[nm][j]
            fresh[nm][j] = need[nm][j] - carried[nm][j]

    # register budget: window elements + outputs + addressing; decides how many CTAs we ask ptxas to fit per SM
    words = sum(len({(u[1], c) for u in held[f.name][j] for c in
                     (range(u[2] * geo[f.name]['vec'], (u[2] + 1) * geo[f.name]['vec']) if u[0] == 'U' else [u[2]])})
                * geo[f.name]['ww'] for f in tma_fields for j in range(D + 1))
    words += sum(SX * (np.dtype(ir.compute_dtype).itemsize if half else lhs.field.dtype.itemsize) // 4 for lhs, _ in ir.main)
    words += sum((qc['hi'] - qc['lo'] + 1) * RY * SX * (np.dtype(ir.compute_dtype).itemsize // 4) for qc in q_classes)
    est_regs = min(255, words + 48)
    # ptxas budgets registers for the CTA size rounded up to 4 warps; a tile whose window cannot fit would spill
    reg_cap = min(255, 65536 // (-(-(THREADS + 32) // 128) * 128))
    if words + 24 > reg_cap and not (t.ty or t.ry):
        raise ValueError('register window of ~%d words does not fit %d threads (cap %d registers)' % (words, THREADS + 32, reg_cap))

    # The window is addressed by *physical* plane slot k = (plane index) mod NP.  In phase PH = step mod NP the
    # plane at stencil position j lives in slot (PH + j + 1) mod NP, so nothing has to be moved between steps: the
    # step body is emitted NP times, once per phase, with the slot numbers baked in.
    any_carry = any(carried[f.name][j] for f in tma_fields for j in range(D + 1)) or bool(q_classes)
    NP = D + 1 if any_carry else 1
    phase = [0]

    def arr(f, j, row):
        g = geo[f.name]
        k = (phase[0] + j + 1) % NP if NP > 1 else j
        return 'R.f%d_k%d_r%d' % (g['ti'], k, row + g['hy'][0])

    def elem(f, j, row, c):
        return '%s[%d]' % (arr(f, j, row), c + geo[f.name]['hx'][0])

    lds_pair = bool(t.lds_pair) and any(
        geo[f.name]['nv'] == 2 and geo[f.name]['es'] == 8 for f in tma_fields)
    # ---- source -------------------------------------------------------------------------------------------------
    jrel = min([j for j in range(D + 1) if any(fresh[f.name][j] for f in tma_fields)] or [D])
    # ring = planes still read from shared memory (D - jrel + 1) + `lookahead` planes in flight ahead of them
    lookahead = t.lookahead or (3 if max_esize <= 4 else 4)   # measured optima (fp32 3-D: sharp at 3; fp64 27-pt: 4)
    STAGES = t.stages or (D - jrel + 1 + max(1, lookahead))
    if STAGES < D - jrel + 2:
        raise ValueError('ring too small')
    smem_bytes = STAGES * STAGE_BYTES + 16 * STAGES
    if smem_bytes > 227 * 1024:
        raise ValueError('ring does not fit in shared memory (%d bytes)' % smem_bytes)
    min_ctas = t.min_ctas or max(1, min(2048 // (THREADS + 32), (227 * 1024) // smem_bytes, 65536 // ((THREADS + 32) * est_regs)))
    out_fields = ir.output_fields
    L = _header(ir, 'march')
    if t.store_mode != 1:
        L.append('#define PSAD_STORE_MODE %d' % t.store_mode)
    L += ['#include "psad_common.cuh"'] + (['#include "%s"' % HALF_HEADER] if half else [])
    L += ['', 'typedef %s CT;' % CT, 'namespace cfg {',
          'constexpr int NDIM = %d, TX = %d, TY = %d, TXS = %d, XORG = 0, TYS = %d, YORG = 0;' % (nd, TX, TY, TX, TY),
          'constexpr int THREADS = %d, MIN_CTAS = %d, STAGES = %d, HZL = %d, HZH = %d, JREL = %d, NP = %d;'
          % (THREADS, min_ctas, STAGES, HZL, HZH, jrel, NP),
          'constexpr int NTMA = %d, STAGE_BYTES = %d, TX_BYTES = %d;' % (len(tma_fields), STAGE_BYTES,
                                                                         sum(geo[f.name]['bytes'] for f in tma_fields)),
          '__device__ constexpr int F_OFF[NTMA] = {%s};' % ', '.join(str(geo[f.name]['off']) for f in tma_fields),
          '__device__ constexpr int F_ORGX[NTMA] = {%s};' % ', '.join(str(-geo[f.name]['padl']) for f in tma_fields),
          '__device__ constexpr int F_ORGY[NTMA] = {%s};' % ', '.join(str(-geo[f.name]['hy'][0]) for f in tma_fields),
          '}  // namespace cfg', '']
    # carry struct: register window + per-item masks / row pointers
    L.append('struct PsadCarry {')
    for f in tma_fields:
        g = geo[f.name]
        W = g['hx'][0] + SX + g['hx'][1]
        if NP > 1:
            all_rows = sorted({u[1] for j in range(D + 1) for u in held[f.name][j]})
            for k in range(NP):
                for row in all_rows:
                    L.append('  %s f%d_k%d_r%d[%d];  // %s, window slot %d, row %+d' % (g['Tw'], g['ti'], k, row + g['hy'][0], W,
                                                                                     f.name, k, row))
        else:
            for j, row in sorted({(j, u[1]) for j in range(D + 1) for u in held[f.name][j]}):
                L.append('  %s f%d_k%d_r%d[%d];  // %s, plane %+d, row %+d' % (g['Tw'], g['ti'], j, row + g['hy'][0], W, f.name,
                                                                            j - HZL, row))
    for ci, qc in enumerate(q_classes):
        for k in range(D + 1):
            for r in range(RY):
                L.append('  CT q%d_k%d_r%d[%d];  // plane sum %d (planes %s), window slot %d, row %d' % (ci, k, r, SX, ci,
                                                                                                  qc['members'], k, r))
    L.append('  unsigned xmask, ymask_wr, ymask_it;  // per item: cells of this thread inside the iteration / write range')
    L.append('  int xs, zlo, zhi;')
    for f in out_fields:
        L.append('  %s* o%d;  // %s: this thread\'s first cell at z = 0' % (_CT[f.dtype.numpy_dtype], fidx[f.name], f.name))
    L.append('};')
    L.append('')
    L.append('PSAD_DEV void psad_item_begin(const PsadArgs& A, PsadCarry& R, int lane, int wy, int y0, int x0)')
    L.append('{')
    L.append('  const int xs = x0 + lane * %d;' % SX)
    L.append('  const int ys = y0 + wy * %d;' % RY)
    L.append('  R.xs = xs;')
    L.append('  R.zlo = (int)A.it_lo[0];')
    L.append('  R.zhi = (int)A.it_hi[0];')
    L.append('  unsigned xm = 0, ymw = 0, ymi = 0;')
    L.append('#pragma unroll')
    L.append('  for (int c = 0; c < %d; ++c) xm |= (xs + c >= (int)A.it_lo[2] && xs + c < (int)A.it_hi[2]) ? (1u << c) : 0u;' % SX)
    L.append('#pragma unroll')
    L.append('  for (int r = 0; r < %d; ++r) {' % RY)
    L.append('    ymw |= (ys + r >= (int)A.wr_lo[1] && ys + r < (int)A.wr_hi[1]) ? (1u << r) : 0u;')
    L.append('    ymi |= (ys + r >= (int)A.it_lo[1] && ys + r < (int)A.it_hi[1]) ? (1u << r) : 0u;')
    L.append('  }')
    L.append('  R.xmask = xm; R.ymask_wr = ymw; R.ymask_it = ymi;')
    for f in out_fields:
        fi = fidx[f.name]
        L.append('  R.o%d = reinterpret_cast<%s*>(A.ptr[%d]) + (long long)ys * A.stride[%d][1] + xs;'
                 % (fi, _CT[f.dtype.numpy_dtype], fi, fi))
    L.append('}')
    L.append('')
    for ph in range(NP):
        phase[0] = ph
        L.append('PSAD_DEV void psad_step_ph%d(const PsadArgs& A, const unsigned char* ring, int slot, PsadCarry& R, int lane,' % ph)
        L.append('                        int wy, bool do_store, int z, int y0, int x0, psad_u32 rel_bar)')
        L.append('{')
        for i, s_ in enumerate(scalars):
            L.append('  const CT %s = (CT)A.scalar[%d];' % (_c_ident(s_), i))
        if lds_pair:
            L.append('  const int lane_hi = (lane >> 2) & 1;')
        for j in range(D + 1):
            if any(fresh[f.name][j] for f in tma_fields):
                back = D - j
                if back == 0:
                    L.append('  const unsigned char* st%d = ring + slot * cfg::STAGE_BYTES;' % j)
                else:
                    L.append('  const unsigned char* st%d = ring + (slot >= %d ? slot - %d : slot - %d + cfg::STAGES) * cfg::STAGE_BYTES;'
                             % (j, back, back, back))
        # fresh loads
        for j in range(D, -1, -1):
            for f in tma_fields:
                g = geo[f.name]
                fr = fresh[f.name][j]
                if not fr:
                    continue
                rows = sorted({u[1] for u in fr})
                for row in rows:
                    rp = 'p%d_%d_%d' % (g['ti'], j, row + g['hy'][0])
                    L.append('  const %s* %s = reinterpret_cast<const %s*>(st%d + %d) + (wy * %d + %d) * %d + %d + lane * %d;'
                             % (g['T'], rp, g['T'], j, g['off'], RY, row + g['hy'][0], g['boxw'], g['padl'], SX))
                    own = sorted(x for x in fr if x[0] == 'U' and x[1] == row)
                    if lds_pair and g['nv'] == 2 and g['es'] == 8 and [u[2] for u in own] == [0, 1]:
                        # both vectors of the 32-byte strip: lane-ordered pair of loads, no bank conflicts
                        L.append('  psad_lds_pair<%s>(%s, lane_hi, &%s);' % (g['T'], rp, elem(f, j, row, 0)))
                        own = []
                    for u in own:
                        if g['es'] == 2:
                            L.append('  psad_lds_h4(%s + %d, &%s);' % (rp, u[2] * g['vec'], elem(f, j, row, u[2] * g['vec'])))
                        else:
                            L.append('  psad_lds_vec<%s>(%s + %d, &%s);' % (g['T'], rp, u[2] * g['vec'], elem(f, j, row, u[2] * g['vec'])))
                    for u in sorted(x for x in fr if x[0] == 'H' and x[1] == row):
                        c = u[2]
                        if t.shuffle:
                            if c < 0:
                                L.append('  %s = psad_from_left(%s);' % (elem(f, j, row, c), elem(f, j, row, src_col(c))))
                                L.append('  if (lane == 0) %s = %s[%d];' % (elem(f, j, row, c), rp, c))
                            else:
                                L.append('  %s = psad_from_right(%s);' % (elem(f, j, row, c), elem(f, j, row, src_col(c))))
                                L.append('  if (lane == 31) %s = %s[%d];' % (elem(f, j, row, c), rp, c))
                        else:
                            L.append('  %s = %s[%d];' % (elem(f, j, row, c), rp, c))
        # this warp will not touch the oldest still-read slot again: hand it back to the producer
        L.append('  __syncwarp();')
        L.append('  if (lane == 0 && rel_bar) psad_mbar_arrive(rel_bar);')
        # plane sums of the plane that just entered the window (needed by later steps: not gated by do_store)
        def qelem(ci, j, r, c):
            return 'R.q%d_k%d_r%d[%d]' % (ci, (phase[0] + j + 1) % NP, r, c)

        def cell_map(r, c):
            # Accesses are first renamed to *absolute* element symbols of the thread's patch (field, plane position,
            # row, column) and only then mapped to registers.  Every sum is ordered by these names, so an expression
            # shared by two cells of the thread (the flux at x-1 of cell x is the flux at x of cell x-1) is printed
            # identically for both and the compiler evaluates it once; the names do not depend on the window phase.
            subs, local = {}, {}
            for f in tma_fields:
                g = geo[f.name]
                for a in raw_accesses[f.name]:
                    dz, dy, dx = _off3(a.offsets)
                    key = sp.Symbol('E%d_%d_%d_%d' % (g['ti'], dz + HZL, r + dy + g['hy'][0], c + dx + g['hx'][0]))
                    subs[a] = key
                    local[key] = '((CT)%s)' % elem(f, dz + HZL, r + dy, c + dx)
            for s_ in ir.scalars:
                local[s_] = _c_ident(s_.name)
            for ci, qc in enumerate(q_classes):
                for dz in qc['members']:
                    local[sp.Symbol('psadQ_%d_%d' % (ci, dz + HZL))] = qelem(ci, dz + HZL, r, c)
            return subs, local

        for hi in sorted({qc['hi'] for qc in q_classes}):
            # all plane sums evaluated at this position, for all cells of the thread, over shared element symbols
            elem_sym, targets = {}, []
            for ci, qc in enumerate(q_classes):
                if qc['hi'] != hi:
                    continue
                for r in range(RY):
                    for c in range(SX):
                        sub = {}
                        for a in qc['expr_hi'].atoms(Field.Access):
                            dz, dy, dx = _off3(a.offsets)
                            g = geo[a.field.name]
                            key = sp.Symbol('E%d_%d_%d' % (g['ti'], r + dy + g['hy'][0], c + dx + g['hx'][0]))
                            elem_sym[key] = '((CT)%s)' % elem(a.field, dz + HZL, r + dy, c + dx)
                            sub[a] = key
                        targets.append(((ci, r, c), qc['expr_hi'].xreplace(sub)))
            plan = plan_linear(targets, set(elem_sym)) if t.linopt else None
            if plan is None:
                for (ci, r, c), _ in targets:
                    subs, local = cell_map(r, c)
                    L.append('  %s = %s;' % (qelem(ci, hi + HZL, r, c),
                                             pr.print_with(q_classes[ci]['expr_hi'].xreplace(subs), local)))
                continue
            txt = {str(k): v for k, v in elem_sym.items()}
            scal = {s_: _c_ident(s_.name) for s_ in ir.scalars}
            L.append('  {')
            for nm, a, b in plan.temps:
                L.append('    const CT %s = %s + %s;' % (nm, txt.get(a, a), txt.get(b, b)))
            for nm, addends in plan.sums:
                parts = [txt.get(a, a) for a in addends]
                while len(parts) > 1:
                    parts = ['(%s + %s)' % (parts[i], parts[i + 1]) if i + 1 < len(parts) else parts[i]
                             for i in range(0, len(parts), 2)]
                L.append('    const CT %s = %s;' % (nm, parts[0]))
            fma = 'fmaf' if CT == 'float' else 'fma'
            for (ci, r, c), lst in plan.targets:
                acc = None
                for coeff, nm in lst:
                    cw = pr.print_with(coeff, scal)
                    acc = '%s * %s' % (cw, txt.get(nm, nm)) if acc is None else '%s(%s, %s, %s)' % (fma, cw, txt.get(nm, nm), acc)
                L.append('    %s = %s;' % (qelem(ci, hi + HZL, r, c), acc))
            L.append('  }')
        # compute + store
        L.append('  if (do_store) {')
        if masked and nd == 3:
            L.append('    const unsigned zm = (z >= R.zlo && z < R.zhi) ? R.ymask_it : 0u;')
        elif masked:
            L.append('    const unsigned zm = R.ymask_it;')
        shared = None
        if cross_cse:
            # One CSE over the inlined right-hand sides of every cell of the thread, in absolute element symbols: what
            # two neighbouring cells have in common (a gradient norm, its reciprocal root, a flux) is evaluated once.
            defs = {}
            for lhs, rhs in ir.subexpressions:
                defs[lhs] = rhs.xreplace(defs)
            all_local, exprs, keys = {}, [], []
            for r in range(RY):
                for c in range(SX):
                    subs, local = cell_map(r, c)
                    # element symbols are absolute (one name per staged value); plane-sum symbols are per cell
                    percell = {k: sp.Symbol('%s_%d_%d' % (k.name, r, c)) for k in local if k.name.startswith('psadQ_')}
                    subs = dict(subs)
                    subs.update(percell)
                    all_local.update({percell.get(k, k): v for k, v in local.items()})
                    for lhs, rhs in main_exprs:
                        exprs.append(_even_power_canonical(rhs.xreplace(defs).xreplace(subs)))
                        keys.append((fidx[lhs.field.name], r, c))
            repl, reduced = sp.cse(exprs, symbols=sp.numbered_symbols('cs'), order='canonical')
            for sym, e in repl:
                L.append('    const CT %s = %s;' % (sym.name, pr.print_with(e, all_local)))
                all_local[sym] = sym.name
            shared = {k: pr.print_with(e, all_local) for k, e in zip(keys, reduced)}
        for r in range(RY):
            L.append('    if ((R.ymask_wr >> %d) & 1u) {' % r)
            if masked:
                L.append('      const unsigned m = ((zm >> %d) & 1u) ? R.xmask : 0u;' % r)
            for lhs, _ in ir.main:
                L.append('      %s o%d[%d];' % (reg_type(lhs.field), fidx[lhs.field.name], SX))
            for c in range(SX):
                if shared is not None:
                    for lhs, _ in main_exprs:
                        To = reg_type(lhs.field)
                        fi = fidx[lhs.field.name]
                        if masked:
                            L.append('      o%d[%d] = ((m >> %d) & 1u) ? (%s)(%s) : (%s)0;' % (fi, c, c, To, shared[(fi, r, c)], To))
                        else:
                            L.append('      o%d[%d] = (%s)(%s);' % (fi, c, To, shared[(fi, r, c)]))
                    continue
                subs, local = cell_map(r, c)
                L.append('      {')
                for lhs, rhs in ir.subexpressions:
                    L.append('        const CT %s = %s;' % (_c_ident(lhs.name), pr.print_with(rhs.xreplace(subs), local)))
                    local[lhs] = _c_ident(lhs.name)
                for lhs, rhs in main_exprs:
                    To = reg_type(lhs.field)
                    text = pr.print_with(rhs.xreplace(subs), local)
                    if masked:
                        L.append('        o%d[%d] = ((m >> %d) & 1u) ? (%s)(%s) : (%s)0;' % (fidx[lhs.field.name], c, c, To, text, To))
                    else:
                        L.append('        o%d[%d] = (%s)(%s);' % (fidx[lhs.field.name], c, To, text))
                L.append('      }')
            for f in out_fields:
                fi = fidx[f.name]
                To = _CT[f.dtype.numpy_dtype]
                vec = vec_cells(f.dtype.itemsize)
                zterm = ' + (long long)z * A.stride[%d][0]' % fi if nd == 3 else ''
                L.append('      %s* q%d = R.o%d%s + %d * A.stride[%d][1];' % (To, fi, fi, zterm, r, fi))
                store = 'psad_stg_h4' if f.dtype.itemsize == 2 else 'psad_stg_vec<%s>' % To
                for v in range(SX // vec):
                    L.append('      if (R.xs + %d <= (int)A.shape[2]) %s(q%d + %d, &o%d[%d]);'
                             % ((v + 1) * vec, store, fi, v * vec, fi, v * vec))
            L.append('    }')
        L.append('  }')
        L.append('}')
        L.append('')
    L.append('PSAD_DEV void psad_step(const PsadArgs& A, const unsigned char* ring, int slot, PsadCarry& R, int lane,')
    L.append('                        int wy, bool do_store, int z, int y0, int x0, psad_u32 rel_bar, int ph)')
    L.append('{')
    if NP == 1:
        L.append('  psad_step_ph0(A, ring, slot, R, lane, wy, do_store, z, y0, x0, rel_bar);')
    else:
        L.append('  switch (ph) {')
        for ph in range(NP):
            L.append('    case %d: psad_step_ph%d(A, ring, slot, R, lane, wy, do_store, z, y0, x0, rel_bar); break;' % (ph, ph))
        L.append('  }')
    L.append('}')
    L.append('')
    L.append('#define PSAD_KERNEL_NAME %s' % name)
    if peer:
        L.append('#define PSAD_PEER 1')
    L.append('#include "psad_march.cuh"')
    L.append('')

    def fplan(f):
        g = geo.get(f.name)
        is_in = f in ir.input_fields
        return dict(elem_size=f.dtype.itemsize, is_input=int(is_in), is_output=int(f in ir.output_fields), index_size=1,
                    tma=int(is_in), box=(g['boxw'], g['boxh'], 1) if is_in else (0, 0, 0))

    plan = dict(kind=1, ndim=nd, n_fields=len(fields), n_scalars=len(scalars), threads=THREADS + 32, smem_bytes=smem_bytes,
                tile_x=TX, tile_y=TY, chunk=t.chunk, ctas_per_sm=t.ctas_per_sm, warmup=D, boundary=1 if ir.boundary == 'zeros' else 0,
                ghost_layers=ir.ghost_layers, peer=int(peer), fields=[fplan(f) for f in fields])
    ek = EmittedKernel(name, 'march', '\n'.join(L), ir, fields, scalars, plan)
    ek.masked = masked
    if ir.fast_math:
        ek.options = ek.options + FAST_MATH_OPTIONS
    ek.geometry = dict(TX=TX, TY=TY, RY=RY, SX=SX, STAGES=STAGES, STAGE_BYTES=STAGE_BYTES, HZ=(HZL, HZH),
                       threads=THREADS, min_ctas=min_ctas)
    return ek


def emit_kernel(ir: StencilKernelIR, variant='auto', tuning=None) -> EmittedKernel:
    if variant == 'generic':
        return emit_generic(ir)
    if variant == 'march':
        return emit_march(ir, tuning)
    if march_ineligible_reason(ir) is None:
        try:
            return emit_march(ir, tuning)
        except ValueError:
            pass
    return emit_generic(ir)
