"""Random stencil generators shared by the CPU (compile-only / replay) and GPU (parity) fuzz tests — any stencil
(``random_stencil``) and one-field stencils for fused pairs of steps (``random_pair_stencil``) — and the per-cell check of
16-bit outputs against the fp64 oracle."""
import random

import numpy as np
import sympy as sp

import pystencils_autodiff_b200 as ps
from oracle.evaluate import evaluate

# x extents for 2-byte fields, by the extent drawn for fp32 / fp64: 136 (a ragged second 128-cell tile), 264 and 40 give
# 16-byte rows and take the march kernel; 36 (72-byte rows) takes the generic kernel only
HALF_X = {132: 136, 128: 264, 64: 40, 36: 36}
MIXED_TYPES = ('float16', 'bfloat16', 'float32')


def random_stencil(seed, shape=None, dtype=None, mixed=False):
    """``(assignments, boundary_handling, shape, dtype)`` of random stencil ``seed``.

    ``dtype`` overrides the drawn field type, ``mixed=True`` gives each field its own type from ``MIXED_TYPES`` (returned
    dtype ``'mixed'``).  Both are applied after every draw, so the stencil and the boundary mode do not depend on them; a
    2-byte ``dtype`` maps a drawn x extent through ``HALF_X``.  With ``boundary_handling=None`` a drawn extent of at most
    twice the ghost layers (no interior cell) grows to ``2 * ghost_layers + 3``; a ``shape`` passed in is kept."""
    rnd = random.Random(seed)
    ndim = rnd.choice([2, 3, 3])
    drawn_dtype = rnd.choice(['float32', 'float64'])
    drawn_shape = shape is None
    if shape is None:
        shape = {2: (rnd.choice([17, 40]), rnd.choice([132, 128, 36])),
                 3: (rnd.choice([5, 9]), rnd.choice([11, 24]), rnd.choice([132, 64, 36]))}[ndim]
    n_in, n_out = rnd.choice([1, 2, 3]), rnd.choice([1, 1, 2])
    names = ['a', 'b', 'c'][:n_in] + ['p', 'q'][:n_out]
    flds = ps.fields('%s: %s[%s]' % (', '.join(names), drawn_dtype, ','.join(map(str, shape))))
    ins, outs = flds[:n_in], flds[n_in:]
    lim = {2: [(-2, 2), (-4, 4)], 3: [(-2, 2), (-2, 2), (-4, 4)]}[ndim]
    narrow = rnd.random() < 0.5

    def access():
        f = rnd.choice(ins)
        off = tuple(rnd.randint(lo, hi) if not narrow else rnd.randint(max(lo, -1), min(hi, 1)) for lo, hi in lim)
        return f[off]

    def term():
        kind = rnd.choice(['lin', 'lin', 'lin', 'prod', 'exp', 'sqrt', 'sin'])
        c = sp.Float(round(rnd.uniform(-1.5, 1.5), 3))
        if kind == 'lin':
            return c * access()
        if kind == 'prod':
            return c * access() * access()
        if kind == 'exp':
            return c * sp.exp(-access() ** 2)
        if kind == 'sqrt':
            return c * access() / sp.sqrt(access() ** 2 + 1)
        return c * sp.sin(access())

    asg = {}
    for o in outs:
        asg[o.center] = sp.Add(*[term() for _ in range(rnd.randint(2, 6))])
    bh = rnd.choice([None, 'zeros'])

    # overrides, after every draw
    types = [dtype or drawn_dtype] * len(names)
    if mixed:
        mrnd = random.Random('mixed%d' % seed)
        types = [mrnd.choice(MIXED_TYPES) for _ in names]
        if len(set(types)) == 1:
            types[-1] = MIXED_TYPES[(MIXED_TYPES.index(types[-1]) + 1) % len(MIXED_TYPES)]
    new_shape = tuple(shape)
    if drawn_shape and dtype in ('float16', 'bfloat16'):
        new_shape = new_shape[:-1] + (HALF_X[new_shape[-1]],)
    if bh is None and drawn_shape:
        gl = max(a.required_ghost_layers for rhs in asg.values() for a in rhs.atoms(ps.Field.Access))
        new_shape = tuple(2 * gl + 3 if n <= 2 * gl else n for n in new_shape)
    if new_shape != tuple(shape) or types != [drawn_dtype] * len(names):
        asg = retyped(asg, new_shape, dict(zip(names, types)))
    return ps.AssignmentCollection(asg), bh, new_shape, 'mixed' if mixed else (dtype or drawn_dtype)


PAIR_SEEDS = range(32)
# reach drawn per side: y / z up to 2, x up to 4 — fp32 strips are 4 cells (two radii beyond a strip need the pad-column
# fix-up loads from 3 cells on), fp64 strips 2 (fix-up loads at 2 cells, no pair beyond)
PAIR_REACH = {'z': (0, 1, 1, 2), 'y': (0, 1, 1, 2), 'x': (0, 1, 2, 2, 3, 4)}


def random_pair_stencil(seed, shape=None):
    """``(assignments, boundary_handling, shape, dtype, scalars)`` of random one-field stencil ``seed`` (``v = S(u)``) for
    fused pairs of steps (emit_chain.py).

    Every term touches one z plane: linear terms, products, ``exp``, ``sqrt`` and ``sin`` of accesses of one plane.  The
    reach is drawn per axis and side (``PAIR_REACH``; one linear term sits at each drawn extreme, so the halo is exactly
    the drawn one); sometimes with an access-free term, sometimes with a symbolic coefficient ``alpha`` whose value is in
    ``scalars``.  2-D stencils have the 'zeros' boundary (the pair runs them lifted to one plane).  Shapes are ragged with
    16-byte rows: y below and above one tile, x a few strips beyond one 120-column tile pitch, z below and above the
    pair's warm-up of 2 x (z reach) planes.  With ``boundary_handling=None`` a drawn extent of at most twice the ghost
    layers grows to ``2 * ghost_layers + 3``; a ``shape`` passed in is kept."""
    rnd = random.Random('pair%d' % seed)
    ndim = rnd.choice([2, 3, 3, 3])
    dtype = rnd.choice(['float32', 'float64'])
    bh = 'zeros' if ndim == 2 else rnd.choice(['zeros', None])
    axes = 'zyx'[3 - ndim:]
    reach = {a: (rnd.choice(PAIR_REACH[a]), rnd.choice(PAIR_REACH[a])) for a in axes}     # (low side, high side)
    nonlinear = rnd.random() < 0.4
    drawn_shape = tuple({'z': rnd.choice([2, 3, 11]), 'y': rnd.choice([13, 50]), 'x': rnd.choice([132, 136, 140])}[a]
                        for a in axes)
    drawn = shape is None
    shape = drawn_shape if drawn else tuple(shape)
    u, v = ps.fields('u, v: %s[%s]' % (dtype, ','.join(map(str, shape))))

    def offset(**fixed):
        return tuple(fixed[a] if a in fixed else rnd.randint(-reach[a][0], reach[a][1]) for a in axes)

    def coeff():
        return sp.Float(round(rnd.choice([-1, 1]) * rnd.uniform(0.2, 1.2), 3))

    def plane_term(kind):
        """A term whose accesses share one z plane."""
        dz = {'z': rnd.randint(-reach['z'][0], reach['z'][1])} if ndim == 3 else {}

        def access():
            return u[offset(**dz)]
        if kind == 'lin':
            return coeff() * access()
        if kind == 'prod':
            return coeff() * access() * access()
        if kind == 'exp':
            return coeff() * sp.exp(-access() ** 2)
        if kind == 'sqrt':
            return coeff() * access() / sp.sqrt(access() ** 2 + 1)
        return coeff() * sp.sin(access())

    terms = []
    for a in axes:                      # the drawn extremes
        for side, r in zip((-1, 1), reach[a]):
            if r:
                terms.append(coeff() * u[offset(**{a: side * r})])
    kinds = ['lin'] * rnd.randint(1, 3)
    if nonlinear:
        kinds += rnd.sample(['prod', 'exp', 'sqrt', 'sin'], rnd.randint(1, 2))
    terms += [plane_term(k) for k in kinds]
    rnd.shuffle(terms)
    scalars = {}
    if rnd.random() < 0.3:
        # a symbolic coefficient of two terms, possibly of different planes: the sum splits by plane only once expanded
        alpha = sp.Symbol('alpha')
        scalars['alpha'] = round(rnd.uniform(0.3, 1.2), 3)
        terms = [alpha * (terms[0] + terms[1])] + terms[2:] if len(terms) > 1 else [alpha * terms[0]]
    if rnd.random() < 0.3:
        terms.append(coeff())           # access-free
    asg = {v.center: sp.Add(*terms)}
    if bh is None and drawn:
        gl = max(a.required_ghost_layers for a in asg[v.center].atoms(ps.Field.Access))
        grown = tuple(2 * gl + 3 if n <= 2 * gl else n for n in shape)
        if grown != shape:
            asg, shape = retyped(asg, grown, dtype), grown
    return ps.AssignmentCollection(asg), bh, shape, dtype, scalars


# ---- one pair fuzz case (shared by the GPU test and its CPU replay) -----------------------------------------------------
def pair_case(seed, shape=None):
    """``(kernels, bh, shape, dtype, scalars)`` of ``random_pair_stencil(seed, shape)``; ``kernels``:
    ``[(direction, ir, assignments)]`` of the forward and — where it reads the upstream gradient only (a linear stencil)
    — the adjoint, the one-field kernels a pair can be asked of."""
    asg, bh, shape, dtype, scalars = random_pair_stencil(seed, shape)
    op = ps.AutoDiffOp(asg, boundary_handling=bh, op_name='pair%d' % seed)
    kernels = [(d, ir, a) for d, ir, a in (('forward', op.forward_ast_gpu, op.forward_assignments),
                                           ('adjoint', op.backward_ast_gpu, op.backward_assignments))
               if len(ir.input_fields) == 1 and len(ir.output_fields) == 1]
    return kernels, bh, shape, dtype, scalars


def pair_input(shape, dtype, seed):
    return np.random.default_rng(seed).uniform(-1, 1, size=shape).astype(dtype)


def oracle_steps(assignments, ir, u, steps, bh, scalars):
    """The fp64 oracle applied ``steps`` times to ``u``, every intermediate result cast to the field type (what a launch
    per step stores); the last result in float64."""
    fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
    r = u
    for i in range(steps):
        r = evaluate(assignments, {fin: r}, bh, scalars=scalars)[fout]
        if i + 1 < steps:
            r = r.astype(u.dtype)
    return r


def check_steps(got, ref, dtype, what=''):
    """Every cell written (no NaN left from the prefilled output), finite, within the fuzz tolerance of the type."""
    got = np.asarray(got, dtype=np.float64)
    assert not np.isnan(got).any(), (what, 'cells not written', int(np.isnan(got).sum()))
    assert np.count_nonzero(ref), (what, 'empty interior')
    scale = max(1.0, np.abs(ref).max())
    err = np.abs(got - ref).max()
    assert np.isfinite(got).all() and err <= WIDE_TOL[dtype] * scale, (what, dtype, err, scale)


def retyped(assignments, shape, types):
    """``{lhs: rhs}`` with every field replaced by one of the same name, of ``shape`` and of type ``types[name]`` (or
    ``types``, one type for all)."""
    def field(name):
        t = types if isinstance(types, str) else types[name]
        return ps.fields('%s: %s[%s]' % (name, t, ','.join(map(str, shape))))

    def swap(e):
        return e.xreplace({a: field(a.field.name)[a.offsets] for a in e.atoms(ps.Field.Access)})
    return {swap(lhs): swap(rhs) for lhs, rhs in assignments.items()}


# ---- 16-bit outputs, cell by cell ----------------------------------------------------------------------------------------
# stored fraction bits, exponent of the smallest normal, exponent of the largest binade
FORMATS = {'float16': (10, -14, 15), 'bfloat16': (7, -126, 127)}
KAPPA = 1e-5            # fp32 arithmetic, relative to max(floor, max |ref|)
KAPPA_DOUBLE = 1e-12    # data_type='double'
WIDE_TOL = {'float32': 2e-5, 'float64': 1e-11}     # wider outputs of mixed kernels: the fuzz tolerance of their type


def spacing(x, dtype):
    """Spacing of ``dtype`` at |x|, subnormal range included."""
    x = np.asarray(x, dtype=np.float64)
    frac, emin, _ = FORMATS[dtype]
    _, e = np.frexp(x)                                # |x| = m 2^e, 1/2 <= m < 1: the binade of x is 2^(e-1)
    return np.ldexp(1.0, np.where(x == 0, emin, np.maximum(e - 1, emin)) - frac)


def round_to(x, dtype):
    """float64 -> nearest ``dtype`` value (ties to even, subnormals, overflow to inf), as float64: ONE rounding, computed
    here in numpy (torch rounds float64 -> bfloat16 through float32, which is two)."""
    x = np.asarray(x, dtype=np.float64)
    q = spacing(x, dtype)
    r = np.round(x / q) * q                           # both exact: q is a power of two
    return np.where(np.abs(r) >= 2.0 ** (FORMATS[dtype][2] + 1), np.copysign(np.inf, x), r)


def to_storage(x, dtype):
    """float64 values -> array as the kernel stores ``dtype`` (bfloat16: raw uint16 words), each value rounded once."""
    with np.errstate(over='ignore'):                  # overflow to inf is what the format does
        if dtype == 'bfloat16':
            return (round_to(x, dtype).astype(np.float32).view(np.uint32) >> 16).astype(np.uint16)
        return np.asarray(x, dtype=np.float64).astype(dtype)


def from_storage(a, dtype):
    """``to_storage`` arrays -> float64, exactly."""
    if dtype == 'bfloat16':
        return (np.asarray(a).view(np.uint16).astype(np.uint32) << 16).view(np.float32).astype(np.float64)
    return np.asarray(a, dtype=np.float64)


def nan_fill(dtype):
    """What outputs are prefilled with: a NaN of ``dtype`` (the bfloat16 word 0x7fc1)."""
    return 0x7fc1 if dtype == 'bfloat16' else np.nan


def check_cells(got, ref, dtype, kappa=KAPPA, floor=1.0, what=''):
    """Every cell of ``got`` (float64, widened exactly from ``dtype``) against the fp64 oracle ``ref``.

    16-bit types: where the single rounding of ref overflows, got is that infinity; elsewhere got is finite and
    |got - ref| <= spacing(ref) / 2 + kappa * max(floor, max |ref|): the one rounding of the stored cell, plus the error of
    the arithmetic before it (``floor``: the scale of the inputs the output is linear in).  Wider types: the fuzz
    tolerance of their type, norm-wise."""
    assert not np.isnan(got).any(), ('NaN (unwritten or invalid) cells', what, int(np.isnan(got).sum()))
    if dtype not in FORMATS:
        scale = max(1.0, np.abs(ref).max())
        assert np.isfinite(got).all() and np.abs(got - ref).max() <= WIDE_TOL[dtype] * scale, (what, dtype)
        return
    r = round_to(ref, dtype)
    over = np.isinf(r)
    assert np.array_equal(got[over], r[over]), ('cells that overflow', what, int((got[over] != r[over]).sum()))
    fin = ~over
    assert np.isfinite(got[fin]).all(), ('inf where the rounded reference is finite', what)
    if not fin.any():
        return
    scale = max(floor, np.abs(ref[fin]).max())
    err = np.abs(np.where(fin, got, 0.0) - np.where(fin, ref, 0.0))
    bound = 0.5 * spacing(ref, dtype) + kappa * scale
    bad = err > bound
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, err / bound, 0)), err.shape)
        raise AssertionError('%s %s: %d of %d cells off; worst at %s: got %r, ref %r, error %.3g spacings (bound %.3g)'
                             % (what, dtype, int(bad.sum()), bad.size, i, got[i], ref[i],
                                err[i] / spacing(ref[i], dtype), bound[i] / spacing(ref[i], dtype)))


# ---- one 16-bit fuzz case: op, fp64 twin, inputs, checks (shared by the GPU test and its CPU replay) -------------------
def field_type(f):
    from pystencils_autodiff_b200.field import BFLOAT16
    return 'bfloat16' if f.dtype.numpy_dtype == BFLOAT16 else np.dtype(f.dtype.numpy_dtype).name


def fuzz_case(seed, dtype=None, mixed=False, shape=None, **op_kwargs):
    """``(op, kernels, bh, shape)`` of random stencil ``seed`` with the type override; ``kernels``:
    ``[(ir, fp64 assignments of the same stencil)]`` for the forward and the adjoint.  The oracle evaluates the float64
    twin: given 16-bit fields it would round its results to them."""
    asg, bh, shape, _ = random_stencil(seed, shape, dtype, mixed)
    op = ps.AutoDiffOp(asg, boundary_handling=bh, op_name='fuzz%d' % seed, **op_kwargs)
    twin = ps.AutoDiffOp(ps.AssignmentCollection(retyped({e.lhs: e.rhs for e in asg.main_assignments}, shape, 'float64')),
                         boundary_handling=bh, op_name='fuzz%d' % seed)
    return op, [(op.forward_ast_gpu, twin.forward_assignments), (op.backward_ast_gpu, twin.backward_assignments)], bh, shape


def fuzz_inputs(fields, ir, shape, seed, diff_scale=1.0):
    """Arrays of ``fields`` as stored (bfloat16: uint16 words): inputs uniform in [-1, 1) (gradient fields ``diff*`` times
    ``diff_scale``), outputs NaN; and the exact float64 values of the inputs."""
    rng = np.random.default_rng(seed)
    stored, values = {}, {}
    for f in fields:
        t = field_type(f)
        if f in ir.input_fields:
            v = rng.uniform(-1, 1, size=shape) * (diff_scale if f.name.startswith('diff') else 1.0)
            stored[f.name] = to_storage(v, t)
            values[f.name] = from_storage(stored[f.name], t)
        else:
            stored[f.name] = np.full(shape, nan_fill(t), dtype=np.uint16 if t == 'bfloat16' else t)
    return stored, values


def ragged_range(shape, gl):
    """A launch range that selects the masked march instance: the write range is wider than the iteration range on every
    side (one cell; in x the whole row, which march kernels write), and the iteration range's x bounds are not multiples
    of 4, so the x mask cuts inside a lane's vector.  Iterated cells keep ``gl`` cells to the array edge (for
    ``boundary_handling=None`` they are interior cells)."""
    it_lo = [gl + 1] * len(shape)
    it_hi = [n - gl - 1 for n in shape]
    while it_lo[-1] % 4 == 0:
        it_lo[-1] += 1
    while it_hi[-1] % 4 == 0:
        it_hi[-1] -= 1
    return dict(iter_lo=it_lo, iter_hi=it_hi, write_lo=[v - 1 for v in it_lo[:-1]] + [0],
                write_hi=[v + 1 for v in it_hi[:-1]] + [shape[-1]])


def check_outputs(ir, stored, ref, launch_range=None, kappa=KAPPA, floor=1.0, what=''):
    """Every output of ``ir`` in ``stored`` against the oracle results ``ref``, in the output's own type (``check_cells``).
    With ``launch_range``: iterated cells as ref, the other written cells 0, cells outside the write range untouched."""
    for f in ir.output_fields:
        t = field_type(f)
        got, r = from_storage(stored[f.name], t), ref[f.name]
        assert np.count_nonzero(r), (what, f.name, 'empty interior')
        name = '%s %s' % (what, f.name)
        if launch_range is None:
            check_cells(got, r, t, kappa, floor, name)
            continue
        it, wr = np.zeros(r.shape, bool), np.zeros(r.shape, bool)
        it[tuple(slice(lo, hi) for lo, hi in zip(launch_range['iter_lo'], launch_range['iter_hi']))] = True
        wr[tuple(slice(lo, hi) for lo, hi in zip(launch_range['write_lo'], launch_range['write_hi']))] = True
        check_cells(got[it], r[it], t, kappa, floor, name)
        assert np.all(got[wr & ~it] == 0), (name, 'written, not iterated cells must be 0')
        assert np.isnan(got[~wr]).all(), (name, 'cells outside the write range must stay untouched')


# adjoints with the upstream gradient scaled by ``scale`` (the adjoint is linear in it): fp16 results in the subnormal
# range and beyond 65504, bf16 results on both sides of fp32's smallest normal and around 1e30
SCALED = [('float16', 1, 1e-6), ('float16', 9, 6e4), ('bfloat16', 1, 1e-37), ('bfloat16', 9, 1e30)]

# data_type='double' cases, by ndim: about 5e5 cells per output, so that results whose rounding through fp32 would land on a
# 16-bit tie and then round the other way (about 2^-14 of the cells for fp16, 2^-17 for bf16) occur
DOUBLE_SHAPES = {2: (2000, 264), 3: (24, 160, 136)}


def reached(dtype, scale, refs):
    """The oracle results of a scaled case are in the edge range it was scaled into."""
    r = np.abs(np.concatenate([a.ravel() for a in refs]))
    r = r[r > 0]
    if dtype == 'float16' and scale < 1:
        assert np.mean(r < 2.0 ** -14) > 0.5                          # mostly fp16 subnormals
    elif dtype == 'float16':
        assert (r >= 65520).any() and (r < 65504).any()               # some overflow, some do not
    elif scale < 1:
        assert (r < 2.0 ** -126).any() and (r >= 2.0 ** -126).any()   # both sides of fp32's smallest normal
    else:
        assert r.max() > 1e30
