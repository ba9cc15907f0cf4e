"""Two applications of one stencil in a single march launch (temporal blocking of unrolled steps).

Reference context: the unrolled time loops of the reference apply the same generated kernel T times and swap
buffers in between (`graph_datahandling.py:152-194,329-344`, `timeloop_astnodes.py:68-145`); every application reads
and writes the whole field in HBM.  SURVEY.md §8 f-1 names fusing steps as the first thing to build after the single
kernel is at the roofline.  This emitter produces, for ``out = S(u)``, a kernel that computes ``out = S(S(u))`` with
the per-step boundary semantics of two separate launches, reading ``u`` once and writing ``out`` once.

How (all inside the march template, `csrc/kernels/psad_march.cuh`):

* the march along z is unchanged; the staged box carries the extra halo the second application needs;
* **stage 1** — when input plane P arrives, every thread evaluates the in-plane groups of the stencil sum for its own
  SX columns and adds them into per-cell accumulators of the intermediate planes in flight.  Plane ``P - HZH`` of the
  intermediate field T is then complete.  T is forced to 0 outside the iteration range — that is what the second
  launch would have read there;
* the T rows stage 2 needs from the neighbouring warps (the y halo) are either **exchanged** — every warp stores its rows
  of the completed plane to a shared buffer, the consumer warps meet at one named barrier, each thread loads the rows
  above and below its own (``MarchTuning.exchange``, default for 4-byte fields; tiles then overlap along y because the
  tile's outermost rows have no owner) — or **recomputed**: stage 1 also covers the halo rows of every thread, and the
  warps never synchronise beyond the TMA ring;
* **stage 2** — the completed T plane is treated exactly like an arriving input plane: x halos come from the
  neighbouring lanes by warp shuffle, the in-plane groups go into the accumulators of the output planes in flight, and
  output plane ``P - 2 HZH`` is complete and stored;
* lanes at the edge of a tile row have no neighbour to take the T halo from, so their columns are not stored: tiles
  overlap by one strip per side (tile pitch ``TXS = 30 * SX`` for a 32-lane row, origin ``XORG = -SX``).

Accumulators are addressed by physical slot ``(phase + k) mod NP`` like the register window of the single-step
kernels, so nothing moves between steps.  Sums are fixed FMA chains (`-fmad=false`), ordered by canonical element
names, hence independent of tiling.
"""
from typing import Optional

import numpy as np
import sympy as sp

from pystencils_autodiff_b200.emit import (FAST_MATH_OPTIONS, EmittedKernel, MarchTuning, _c_ident, _CT,
                                           _CudaPrinter, _header, _kernel_name, _off3, march_ineligible_reason)
from pystencils_autodiff_b200.field import Field
from pystencils_autodiff_b200.ir import StencilKernelIR
from pystencils_autodiff_b200.linopt import plan_linear

__all__ = ['chain_ineligible_reason', 'emit_march_chain']


def chain_ineligible_reason(ir: StencilKernelIR) -> Optional[str]:
    if any(f.dtype.numpy_dtype == np.dtype(np.float16) for f in ir.all_fields):
        # a pair would carry the intermediate field in fp32 and round once, two launches round it to fp16 in between
        return 'float16 fields: fused pairs not implemented'
    reason = march_ineligible_reason(ir)
    if reason:
        return reason
    if ir.ndim != 3:
        return 'step fusion is implemented for 3-D fields'
    if len(ir.main) != 1 or ir.subexpressions:
        return 'step fusion needs a single assignment without subexpressions'
    if len(ir.input_fields) != 1 or len(ir.output_fields) != 1:
        return 'step fusion needs one input and one output field'
    fin, fout = ir.input_fields[0], ir.output_fields[0]
    if fin.dtype.numpy_dtype != fout.dtype.numpy_dtype:
        return 'input and output must have the same element type'
    if _planewise(ir.main[0][1]) is None:
        return 'a term couples several z planes'
    return None


def _planewise(rhs):
    """``rhs`` as a sum whose terms each touch one z plane (expanded if the given form does not split), else None."""
    for cand in (rhs, sp.expand(rhs)):
        if all(len({int(a.offsets[0]) for a in term.atoms(Field.Access)}) <= 1 for term in sp.Add.make_args(cand)):
            return cand
    return None


def emit_march_chain(ir: StencilKernelIR, tuning: Optional[MarchTuning] = None, peer: bool = False) -> EmittedKernel:
    """Kernel computing ``out = S(S(u))`` for the single-step IR ``out = S(u)`` (fields: out, u)."""
    reason = chain_ineligible_reason(ir)
    if reason:
        raise ValueError('fused-step march variant not applicable: ' + reason)
    t = tuning or MarchTuning()
    CT = _CT[ir.compute_dtype]
    pr = _CudaPrinter(ir.compute_dtype)
    fin, fout = ir.input_fields[0], ir.output_fields[0]
    fields = ir.all_fields                     # (out, u)
    fidx = {f.name: i for i, f in enumerate(fields)}
    scalars = [s.name for s in ir.scalars]
    es = fin.dtype.itemsize
    T = _CT[fin.dtype.numpy_dtype]
    vec = 16 // es

    # ---- geometry ------------------------------------------------------------------------------------------------
    (HZL, HZH), (HYL, HYH), (HXL, HXR) = [tuple(h) for h in ir.halo(fin.name)]
    D1 = HZL + HZH
    # measured on B200 (scripts/steps_bench.py), 7-point fp32 at 1024^3, two launches = 2.77 ms:
    #   rows exchanged through shared memory, 44x128 tiles, 4 x 4 cells per thread, 11+1 warps, 168 registers: 1.73 ms
    #   same with 30x128 tiles, 2 x 4 cells, 15+1 warps, 109 registers: 1.79 ms
    #   rows recomputed, 30x128 tiles, 2 x 4 cells, 15+1 warps, 128 registers: 1.99 ms
    # 27-point fp64 at 768^3, two launches = 2.31 ms (round 2, scripts/steps_bench.py): recomputed rows 22x64 / 2 x 2 cells /
    # 11+1 warps 2.28 ms; exchanged rows 28x64 / 4 x 2 cells, one CTA per SM 2.37 ms; exchanged rows with TWO CTAs per SM
    # (while one waits at its per-plane barrier the other computes) 18x64 tiles / 2 x 2 cells / 9+1 warps / 96 registers:
    # 2.09 ms = 1.11x — the fp64 default; 14x64: 2.12 ms, three CTAs of 10x64: 2.64 ms.
    want_exchange = True if t.exchange is None else bool(t.exchange)
    fp64_default = es == 8 and want_exchange and not (t.ry or t.ty or t.sx or t.min_ctas)
    if fp64_default:
        import dataclasses
        t = dataclasses.replace(t, ry=2, ty=18, sx=2, min_ctas=2)
    SX = t.sx or (4 if es == 4 else 2)
    if (SX * es) % 16:
        raise ValueError('sx*itemsize must be a multiple of 16 bytes')
    if HXL > SX or HXR > SX:
        raise ValueError('x halo wider than the per-thread strip')
    RY = t.ry or (4 if (es == 4 and want_exchange) else 2)
    # warps: the register budget is per CTA size rounded up to 4 warps (11+1 warps: 170 registers, 15+1: 128)
    TY = t.ty or (RY * (11 if (es == 8 or want_exchange) else 15))
    if TY % RY:
        raise ValueError('ty must be a multiple of ry')
    THREADS = 32 * (TY // RY)
    if THREADS + 32 > 1024:
        raise ValueError('tile too tall: %d threads' % THREADS)
    TX = 32 * SX
    EL, ER = int(HXL > 0), int(HXR > 0)            # edge lanes whose columns cannot be completed
    TXS = (32 - EL - ER) * SX
    XORG = -EL * SX
    # The input halo of the row's first / last lane would have to come from shared memory (pad columns in the box).
    # Those lanes are not stored, and what their neighbours take from them — the T columns next to the lane border —
    # does not depend on that halo as long as two radii fit into one strip: then no pad columns and no fix-up loads.
    fixup = 2 * HXL > SX or 2 * HXR > SX
    padl = -(-HXL // vec) * vec if fixup else 0
    padr = -(-HXR // vec) * vec if fixup else 0
    boxw = TX + padl + padr
    # Intermediate rows owned by the neighbouring warps: recomputed by every thread (input box with two y radii), or —
    # `exchange` — written to a shared buffer by their owners and read back after one consumer barrier (input box with
    # one y radius; the tile's outermost rows have no owner, so tiles then overlap along y as well)
    exchange = want_exchange and D1 > 0 and HYL + HYH > 0      # needs >= 2 window phases; pointless without a y halo
    name = _kernel_name(ir, ('march_x2e' if exchange else 'march_x2') + ('_peer' if peer else ''))
    U_L, U_H = (HYL, HYH) if exchange else (2 * HYL, 2 * HYH)      # input rows above / below the thread's own rows
    TYS = TY - HYL - HYH if exchange else TY
    YORG = -HYL if exchange else 0
    if TYS < 1:
        raise ValueError('tile too short for the y halo')
    boxh = TY + U_L + U_H
    if boxw > 256 or boxh > 256:
        raise ValueError('TMA box too large')
    STAGE_BYTES = -(-(boxw * boxh * es) // 128) * 128
    lookahead = t.lookahead or (3 if es == 4 else 4)
    STAGES = t.stages or (1 + max(1, lookahead))
    if STAGES < 2:
        raise ValueError('ring too small')
    NP = D1 + 1
    cwb = np.dtype(ir.compute_dtype).itemsize
    XB_ROWS = TY + HYL + HYH                        # exchange buffer: one intermediate plane of the tile + unowned pad rows
    XBUF_OFF = -(-(STAGES * STAGE_BYTES + 16 * STAGES) // 128) * 128
    smem_bytes = XBUF_OFF + NP * XB_ROWS * TX * cwb if exchange else STAGES * STAGE_BYTES + 16 * STAGES
    if smem_bytes > 227 * 1024:
        raise ValueError('ring does not fit in shared memory (%d bytes)' % smem_bytes)
    rows1 = list(range(0, RY)) if exchange else list(range(-HYL, RY + HYH))   # rows of T a thread evaluates
    trows = list(range(-HYL, RY + HYH))             # rows of T its second stage reads
    rows0 = list(range(-U_L, RY + U_H))             # rows of u it reads
    A1 = -rows1[0]                                  # row offset of the stage-1 accumulator / mask arrays
    cw = np.dtype(ir.compute_dtype).itemsize // 4
    words = (len(rows1) + RY) * SX * cw * D1 + len(rows0) * (SX + HXL + HXR) * (es // 4)
    reg_cap = min(255, 65536 // (-(-(THREADS + 32) // 128) * 128))
    min_ctas = t.min_ctas or max(1, min(2048 // (THREADS + 32), (227 * 1024) // smem_bytes,
                                        65536 // ((THREADS + 32) * min(255, words + 48))))

    # ---- the stencil sum split by plane: rhs = sum_dz G_dz, G grouped by canonical (z-shifted) expression ----------
    rhs = _planewise(ir.main[0][1])

    def zshift(expr, dz):
        return expr.xreplace({a: a.get_shifted(dz, 0, 0) for a in expr.atoms(Field.Access)})

    groups = {}
    const_terms = []
    for term in sp.Add.make_args(rhs):
        dzs = {int(a.offsets[0]) for a in term.atoms(Field.Access)}
        if not dzs:
            const_terms.append(term)
        else:
            groups.setdefault(dzs.pop(), []).append(term)
    if const_terms:
        groups.setdefault(HZH, []).append(sp.Add(*const_terms))     # access-free terms join the completing plane
    canon = []                  # [(expr over accesses at dz = 0, [dz, ...])]
    for dz in sorted(groups):
        c = zshift(sp.Add(*groups[dz]), -dz)
        for entry in canon:
            if entry[0] == c:
                entry[1].append(dz)
                break
        else:
            canon.append((c, [dz]))
    class_of = {dz: ci for ci, (_, dzs) in enumerate(canon) for dz in dzs}

    # ---- source ---------------------------------------------------------------------------------------------------
    L = _header(ir, 'march_x2', '// two applications of the stencil per launch: out = S(S(%s))' % fin.name)
    if t.store_mode != 1:
        L.append('#define PSAD_STORE_MODE %d' % t.store_mode)
    L += ['#include "psad_common.cuh"', '', 'typedef %s CT;' % CT, 'namespace cfg {',
          'constexpr int NDIM = 3, TX = %d, TY = %d, TXS = %d, XORG = %d, TYS = %d, YORG = %d;' % (TX, TY, TXS, XORG, TYS, YORG),
          'constexpr int THREADS = %d, MIN_CTAS = %d, STAGES = %d, HZL = %d, HZH = %d, JREL = %d, NP = %d;'
          % (THREADS, min_ctas, STAGES, 2 * HZL, 2 * HZH, 2 * D1, NP),
          'constexpr int NTMA = 1, STAGE_BYTES = %d, TX_BYTES = %d;' % (STAGE_BYTES, boxw * boxh * es),
          '__device__ constexpr int F_OFF[NTMA] = {0};',
          '__device__ constexpr int F_ORGX[NTMA] = {%d};' % -padl,
          '__device__ constexpr int F_ORGY[NTMA] = {%d};' % -U_L] + \
         (['constexpr int SMEM_BYTES = %d, XBUF_OFF = %d, XB_PLANE = %d;  // exchange buffers: NP planes of %d x TX values'
           % (smem_bytes, XBUF_OFF, XB_ROWS * TX, XB_ROWS)] if exchange else []) + \
         ['}  // namespace cfg', ''] + (['#define PSAD_CTA_EXCHANGE 1', ''] if exchange else [])
    L.append('struct PsadCarry {')
    for k in range(NP):
        for r in rows1:
            L.append('  CT a1_k%d_r%d[%d];  // intermediate plane accumulator, slot %d, row %+d' % (k, r + A1, SX, k, r))
    for k in range(NP):
        for r in range(RY):
            L.append('  CT a2_k%d_r%d[%d];  // output plane accumulator, slot %d, row %d' % (k, r, SX, k, r))
    L.append('  unsigned xmask, ymask_wr, ymask_it, ymask_t;  // per item: cells inside the iteration / write range')
    L.append('  int xs, zlo, zhi;')
    L.append('  %s* o0;  // %s: this thread\'s first cell at z = 0' % (T, fout.name))
    L.append('};')
    L.append('')
    fo = fidx[fout.name]
    L += ['PSAD_DEV void psad_item_begin(const PsadArgs& A, PsadCarry& R, int lane, int wy, int y0, int x0)',
          '{',
          '  const int xs = x0 + lane * %d;' % SX,
          '  const int ys = y0 + wy * %d;' % RY,
          '  R.xs = xs;',
          '  R.zlo = (int)A.it_lo[0];',
          '  R.zhi = (int)A.it_hi[0];',
          '  unsigned xm = 0, ymw = 0, ymi = 0, ymt = 0;',
          '#pragma unroll',
          '  for (int c = 0; c < %d; ++c) xm |= (xs + c >= (int)A.it_lo[2] && xs + c < (int)A.it_hi[2]) ? (1u << c) : 0u;' % SX,
          '#pragma unroll',
          '  for (int r = 0; r < %d; ++r) {' % RY,
          '    ymw |= (ys + r >= (int)A.wr_lo[1] && ys + r < (int)A.wr_hi[1]) ? (1u << r) : 0u;',
          '    ymi |= (ys + r >= (int)A.it_lo[1] && ys + r < (int)A.it_hi[1]) ? (1u << r) : 0u;',
          '  }',
          '#pragma unroll',
          '  for (int r = 0; r < %d; ++r)' % len(rows1),
          '    ymt |= (ys + r - %d >= (int)A.it_lo[1] && ys + r - %d < (int)A.it_hi[1]) ? (1u << r) : 0u;' % (A1, A1),
          # lanes whose columns are recomputed by the neighbouring tile, or lie beyond the row, never store
          '  if (lane < %d || lane >= %d%s) ymw = 0;' % (EL, 32 - ER, ' || xs + %d > (int)A.shape[2]' % SX if SX == vec else '')] + \
         (['#pragma unroll',     # exchange: the tile's outermost rows get no intermediate rows from a neighbour
           '  for (int r = 0; r < %d; ++r)' % RY,
           '    if (wy * %d + r < %d || wy * %d + r >= %d) ymw &= ~(1u << r);' % (RY, HYL, RY, TY - HYH)] if exchange else []) + [
          '  R.xmask = xm; R.ymask_wr = ymw; R.ymask_it = ymi; R.ymask_t = ymt;',
          '  R.o0 = reinterpret_cast<%s*>(A.ptr[%d]) + (long long)ys * A.stride[%d][1] + xs;' % (T, fo, fo),
          '}', '']

    fma = 'fmaf' if CT == 'float' else 'fma'
    scal = {s_: _c_ident(s_.name) for s_ in ir.scalars}

    def fold(contrib, init):
        """Text of ``init + contribution`` (``init`` None: the contribution alone)."""
        kind, val = contrib
        if kind == 'var':
            return val if init is None else '(%s + %s)' % (init, val)
        acc = init
        for cwt, operand in val:
            acc = '%s * %s' % (cwt, operand) if acc is None else '%s(%s, %s, %s)' % (fma, cwt, operand, acc)
        return acc

    def emit_groups(stage, cells, elem_text):
        """Evaluate the canonical in-plane groups for every cell.  Returns {(ci, r, c): contribution}: either
        ('var', name) — the group value, computed once and added wherever it is used — or ('chain', [(w, operand)])
        — a short weighted sum that is cheaper to fold into each accumulator as FMAs than to form and add."""
        out = {}
        elem_sym, targets = {}, []
        for ci, (expr, _) in enumerate(canon):
            for (r, c) in cells:
                sub = {}
                for a in expr.atoms(Field.Access):
                    _, dy, dx = _off3(a.offsets)
                    key = sp.Symbol('E%d_%d_%d' % (stage, r + dy + 2 * HYL, c + dx + HXL))
                    elem_sym[key] = elem_text(r + dy, c + dx)
                    sub[a] = key
                targets.append(((ci, r, c), expr.xreplace(sub)))
        plan = plan_linear(targets, set(elem_sym)) if t.linopt else None
        if plan is None:
            local = dict(scal)
            local.update(elem_sym)
            for key, expr in targets:
                nm = 'g%d_%d_%d_%d' % (stage, key[0], key[1] + HYL, key[2])
                L.append('  const CT %s = %s;' % (nm, pr.print_with(expr, local)))
                out[key] = ('var', nm)
            return out
        txt = {str(k): v for k, v in elem_sym.items()}
        for nm, a, b in plan.temps:
            txt[nm] = 's%d_%s' % (stage, nm)
            L.append('  const CT %s = %s + %s;' % (txt[nm], txt.get(a, a), txt.get(b, b)))
        for nm, addends in plan.sums:
            parts = [txt.get(a, a) for a in addends]
            while len(parts) > 1:
                parts = ['(%s + %s)' % (parts[i], parts[i + 1]) if i + 1 < len(parts) else parts[i]
                         for i in range(0, len(parts), 2)]
            txt[nm] = 's%d_%s' % (stage, nm)
            L.append('  const CT %s = %s;' % (txt[nm], parts[0]))
        for key, lst in plan.targets:
            uses = len(canon[key[0]][1])
            chain = [(pr.print_with(coeff, scal), txt.get(nm, nm)) for coeff, nm in lst]
            if uses * len(chain) < len(chain) + uses:
                out[key] = ('chain', chain)
            else:
                nm = 'g%d_%d_%d_%d' % (stage, key[0], key[1] + HYL, key[2])
                L.append('  const CT %s = %s;' % (nm, fold(('chain', chain), None)))
                out[key] = ('var', nm)
        return out

    def accumulate(stage, ph, cells, contribs, done):
        """Fold the groups of the arriving plane into the accumulators; ``done(r, c, text)`` receives the completed value."""
        def acc(k, r, c):
            return 'R.a%d_k%d_r%d[%d]' % (stage, (ph + k) % NP, r + (A1 if stage == 1 else 0), c)

        for (r, c) in cells:
            for k in range(D1, -1, -1):          # k = D1: first contribution ... k = 0: last one, plane complete
                dz = HZH - k
                g = contribs[(class_of[dz], r, c)] if dz in class_of else None
                if k == D1 and k > 0:
                    L.append('  %s = %s;' % (acc(k, r, c), fold(g, None) if g else '(CT)0'))
                elif k > 0:
                    if g:
                        L.append('  %s = %s;' % (acc(k, r, c), fold(g, acc(k, r, c))))
                elif D1 == 0:
                    done(r, c, fold(g, None) if g else '(CT)0')
                else:
                    done(r, c, fold(g, acc(0, r, c)) if g else acc(0, r, c))

    W0 = HXL + SX + HXR
    for ph in range(NP):
        L.append('PSAD_DEV void psad_step_ph%d(const PsadArgs& A, const unsigned char* ring, int slot, PsadCarry& R, int lane,' % ph)
        L.append('                        int wy, bool do_store, int z, int y0, int x0, psad_u32 rel_bar)')
        L.append('{')
        for i, s_ in enumerate(scalars):
            L.append('  const CT %s = (CT)A.scalar[%d];' % (_c_ident(s_), i))
        L.append('  const unsigned char* st = ring + slot * cfg::STAGE_BYTES;')
        # ---- stage 1: the arriving input plane
        for r in rows0:
            ri = r + U_L
            L.append('  %s u%d[%d];' % (T, ri, W0))
            L.append('  const %s* p%d = reinterpret_cast<const %s*>(st) + (wy * %d + %d) * %d + %d + lane * %d;'
                     % (T, ri, T, RY, ri, boxw, padl, SX))
            for v in range(SX // vec):
                L.append('  psad_lds_vec<%s>(p%d + %d, &u%d[%d]);' % (T, ri, v * vec, ri, HXL + v * vec))
        for r in rows0:
            ri = r + U_L
            for c in range(-HXL, 0):
                L.append('  u%d[%d] = psad_from_left(u%d[%d]);' % (ri, c + HXL, ri, SX + c + HXL))
                if fixup:
                    L.append('  if (lane == 0) u%d[%d] = p%d[%d];' % (ri, c + HXL, ri, c))
            for c in range(SX, SX + HXR):
                L.append('  u%d[%d] = psad_from_right(u%d[%d]);' % (ri, c + HXL, ri, c - SX + HXL))
                if fixup:
                    L.append('  if (lane == 31) u%d[%d] = p%d[%d];' % (ri, c + HXL, ri, c))
        L.append('  __syncwarp();')
        L.append('  if (lane == 0 && rel_bar) psad_mbar_arrive(rel_bar);')
        cells1 = [(r, c) for r in rows1 for c in range(SX)]
        g1 = emit_groups(1, cells1, lambda r, c: '((CT)u%d[%d])' % (r + U_L, c + HXL))
        L.append('  // intermediate plane z + %d is complete; outside the iteration range the next step would read 0' % HZH)
        L.append('  const unsigned tm = (z + %d >= R.zlo && z + %d < R.zhi) ? R.ymask_t : 0u;' % (HZH, HZH))
        for r in trows:
            L.append('  CT t%d[%d];' % (r + HYL, W0))

        def done1(r, c, text):
            L.append('  t%d[%d] = %s;' % (r + HYL, c + HXL, text))
        accumulate(1, ph, cells1, g1, done1)
        # only tiles on the boundary of the iteration range (and planes outside it) pay for the selects
        L.append('  if (tm != %du || R.xmask != %du) {' % ((1 << len(rows1)) - 1, (1 << SX) - 1))
        for (r, c) in cells1:
            L.append('    t%d[%d] = (((tm >> %d) & 1u) && ((R.xmask >> %d) & 1u)) ? t%d[%d] : (CT)0;'
                     % (r + HYL, c + HXL, r + A1, c, r + HYL, c + HXL))
        L.append('  }')
        if exchange:
            # own rows -> shared buffer of this phase; barrier over the consumer warps; neighbours' rows <- buffer.  NP >= 2
            # buffers: a warp that is one step ahead writes another buffer than the one a slower warp still reads, and
            # cannot get two steps ahead without that warp passing the next barrier.
            L.append('  CT* xb = reinterpret_cast<CT*>(const_cast<unsigned char*>(ring) + cfg::XBUF_OFF) + %d * cfg::XB_PLANE'
                     ' + (wy * %d + %d) * %d + lane * %d;' % (ph, RY, HYL, TX, SX))
            cvec = 16 // cwb
            for r in rows1:
                for v in range(SX // cvec):
                    L.append('  psad_sts_vec<CT>(xb + %d + %d, &t%d[%d]);' % (r * TX, v * cvec, r + HYL, HXL + v * cvec))
            L.append('  psad_consumer_barrier(cfg::THREADS);')
            for r in trows:
                if r in rows1:
                    continue
                for v in range(SX // cvec):
                    L.append('  psad_lds_vec<CT>(xb + (%d) + %d, &t%d[%d]);' % (r * TX, v * cvec, r + HYL, HXL + v * cvec))
        # ---- stage 2: the completed intermediate plane arrives
        for r in trows:
            ri = r + HYL
            for c in range(-HXL, 0):
                L.append('  t%d[%d] = psad_from_left(t%d[%d]);' % (ri, c + HXL, ri, SX + c + HXL))
            for c in range(SX, SX + HXR):
                L.append('  t%d[%d] = psad_from_right(t%d[%d]);' % (ri, c + HXL, ri, c - SX + HXL))
        cells2 = [(r, c) for r in range(RY) for c in range(SX)]
        g2 = emit_groups(2, cells2, lambda r, c: 't%d[%d]' % (r + HYL, c + HXL))
        for r in range(RY):
            L.append('  CT v%d[%d];' % (r, SX))

        def done2(r, c, text):
            L.append('  v%d[%d] = %s;' % (r, c, text))
        accumulate(2, ph, cells2, g2, done2)
        L.append('  if (do_store && R.ymask_wr) {')
        L.append('    const unsigned zm = (z >= R.zlo && z < R.zhi) ? R.ymask_it : 0u;')
        for r in range(RY):
            L.append('    if ((R.ymask_wr >> %d) & 1u) {' % r)
            L.append('      const unsigned m = ((zm >> %d) & 1u) ? R.xmask : 0u;' % r)
            L.append('      %s o[%d];' % (T, SX))
            for c in range(SX):
                L.append('      o[%d] = (%s)v%d[%d];' % (c, T, r, c))
            L.append('      if (m != %du) {' % ((1 << SX) - 1))
            for c in range(SX):
                L.append('        if (!((m >> %d) & 1u)) o[%d] = (%s)0;' % (c, c, T))
            L.append('      }')
            L.append('      %s* q = R.o0 + (long long)z * A.stride[%d][0] + %d * A.stride[%d][1];' % (T, fo, r, fo))
            for v in range(SX // vec):
                guard = 'if (R.xs + %d <= (int)A.shape[2]) ' % ((v + 1) * vec) if SX != vec else ''
                L.append('      %spsad_stg_vec<%s>(q + %d, &o[%d]);' % (guard, T, v * vec, v * vec))
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
        L.append('#define PSAD_PEER 1      // ghost planes from the neighbouring GPUs\' arrays (psad_kernel_launch_peer)')
    L.append('#include "psad_march.cuh"')
    L.append('')

    def fplan(f):
        is_in = f is fin
        return dict(elem_size=f.dtype.itemsize, is_input=int(is_in), is_output=int(f is fout), index_size=1,
                    tma=int(is_in), box=(boxw, boxh, 1) if is_in else (0, 0, 0))

    plan = dict(kind=1, ndim=3, n_fields=len(fields), n_scalars=len(scalars), threads=THREADS + 32, smem_bytes=smem_bytes,
                tile_x=TXS, tile_y=TYS, chunk=t.chunk, ctas_per_sm=t.ctas_per_sm, warmup=2 * D1, fused_steps=2,
                boundary=1 if ir.boundary == 'zeros' else 0, ghost_layers=ir.ghost_layers, peer=int(peer),
                fields=[fplan(f) for f in fields])
    ek = EmittedKernel(name, 'march', '\n'.join(L), ir, fields, scalars, plan)
    ek.masked = True
    if ir.fast_math:
        ek.options = ek.options + FAST_MATH_OPTIONS
    ek.geometry = dict(TX=TX, TY=TY, RY=RY, SX=SX, TXS=TXS, TYS=TYS, exchange=exchange, STAGES=STAGES, STAGE_BYTES=STAGE_BYTES, HZ=(2 * HZL, 2 * HZH),
                       threads=THREADS, min_ctas=min_ctas, reg_cap=reg_cap, est_words=words)
    return ek
