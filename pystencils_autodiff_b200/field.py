"""Minimal stencil front end: ``Field``, ``Field.Access`` and ``fields()``.

The reference builds its operators out of pystencils objects (``pystencils.fields``,
``Field.Access``; used at /root/reference/tests/test_autodiff.py:10,
/root/reference/README.rst:53-57, /root/reference/src/pystencils_autodiff/_autodiff.py:47-52).
pystencils is a third-party dependency that is not part of the reference tree, so this module
provides the small subset of that API the ``torch_native`` path touches.  Objects coming from
a real pystencils installation are accepted everywhere through :func:`coerce_access`, which
only relies on the duck-typed attributes ``field``, ``offsets``, ``index``, ``name``, ``dtype``
and ``spatial_shape``.

Access naming (``x_C``, ``x_E``, ``x_2W`` ...) follows the reference's printed known answers
(/root/reference/tests/test_autodiff.py:21, /root/reference/README.rst:66-68,85-86).
"""
import re
from typing import Sequence, Tuple

import numpy as np
import sympy as sp

__all__ = ['Field', 'FieldType', 'BasicType', 'fields', 'coerce_access', 'coerce_field',
           'offset_to_direction_string', 'x_vector', 'BFLOAT16']

# numpy has no bfloat16: bfloat16 fields carry this 2-byte stand-in as their numpy dtype.  Their values only ever live in
# torch.bfloat16 tensors; host copies (gather_array, save_fields) are widened to float32.
BFLOAT16 = np.dtype([('bfloat16', '<u2')])

_C_TYPE_NAMES = {
    'double': np.float64, 'float': np.float32, 'float64': np.float64, 'float32': np.float32,
    'int': np.int32, 'int32': np.int32, 'int64': np.int64, 'float16': np.float16, 'bfloat16': BFLOAT16,
}


class FieldType:
    GENERIC = 0
    INDEXED = 1
    BUFFER = 3
    CUSTOM = 4


class BasicType:
    """dtype wrapper exposing ``numpy_dtype`` like pystencils' ``BasicType``."""

    def __init__(self, dtype):
        if isinstance(dtype, BasicType):
            dtype = dtype.numpy_dtype
        elif hasattr(dtype, 'numpy_dtype'):
            dtype = dtype.numpy_dtype
        elif isinstance(dtype, str) and dtype in _C_TYPE_NAMES:
            dtype = _C_TYPE_NAMES[dtype]
        self.numpy_dtype = np.dtype(dtype)

    @property
    def c_name(self):
        return {np.dtype(np.float64): 'double', np.dtype(np.float32): 'float',
                np.dtype(np.int32): 'int', np.dtype(np.int64): 'int64_t',
                np.dtype(np.float16): 'half', BFLOAT16: 'bfloat16'}[self.numpy_dtype]

    @property
    def itemsize(self):
        return self.numpy_dtype.itemsize

    def __eq__(self, other):
        return isinstance(other, BasicType) and self.numpy_dtype == other.numpy_dtype

    def __hash__(self):
        return hash(self.numpy_dtype.str)

    def __str__(self):
        return self.c_name

    __repr__ = __str__


def x_vector(dim):
    """Loop counter symbols ``ctr_0 … ctr_{dim-1}`` (pystencils' ``x_vector``)."""
    return sp.Matrix([sp.Symbol('ctr_%d' % i, integer=True) for i in range(dim)])


def _offset_component(coordinate_id: int, value: int) -> str:
    names = (('W', 'E'), ('S', 'N'), ('B', 'T'))
    if value == 0:
        return ''
    res = names[coordinate_id][0 if value < 0 else 1]
    if abs(value) > 1:
        res = '%d%s' % (abs(value), res)
    return res


def offset_to_direction_string(offsets: Sequence[int]) -> str:
    if len(offsets) > 3:
        return str(tuple(offsets))
    names = [_offset_component(i, int(o)) for i, o in enumerate(offsets)]
    name = ''.join(reversed(names))
    return name if name else 'C'


class Field:
    """A named n-dimensional array with ``index_dimensions`` trailing per-cell components."""

    def __init__(self, name, field_type, dtype, layout, shape, strides=None):
        self.name = name
        self.field_type = field_type
        self._dtype = BasicType(dtype)
        self._layout = tuple(layout)
        self.shape = tuple(shape)
        self.latex_name = None
        if strides is None:
            strides = self._default_strides(self.shape)
        self.strides = tuple(strides)

    # -- construction helpers ------------------------------------------------------------------
    @staticmethod
    def _default_strides(shape):
        if all(isinstance(s, (int, np.integer)) for s in shape):
            st, acc = [], 1
            for s in reversed(shape):
                st.append(acc)
                acc *= int(s)
            return tuple(reversed(st))
        return tuple(sp.Symbol('_stride_%d' % i, integer=True) for i in range(len(shape)))

    @staticmethod
    def create_fixed_size(field_name, shape, index_dimensions=0, dtype=np.float64, layout='numpy',
                          strides=None, field_type=FieldType.GENERIC):
        shape = tuple(int(s) for s in shape)
        spatial = len(shape) - index_dimensions
        f = Field(field_name, field_type, dtype, tuple(range(spatial)), shape, strides)
        f._index_dimensions = index_dimensions
        return f

    @staticmethod
    def create_generic(field_name, spatial_dimensions, dtype=np.float64, index_dimensions=0,
                       layout='numpy', index_shape=None, field_type=FieldType.GENERIC):
        shape = tuple(sp.Symbol('_size_%s_%d' % (field_name, i), integer=True)
                      for i in range(spatial_dimensions))
        if index_shape is None:
            index_shape = tuple(sp.Symbol('_size_%s_%d' % (field_name, spatial_dimensions + i), integer=True)
                                for i in range(index_dimensions))
        shape = shape + tuple(index_shape)
        strides = tuple(sp.Symbol('_stride_%s_%d' % (field_name, i), integer=True) for i in range(len(shape)))
        f = Field(field_name, field_type, dtype, tuple(range(spatial_dimensions)), shape, strides)
        f._index_dimensions = len(index_shape)
        return f

    @staticmethod
    def create_from_numpy_array(field_name, array, index_dimensions=0, field_type=FieldType.GENERIC):
        shape = tuple(int(s) for s in array.shape)
        if hasattr(array, 'strides') and not callable(array.strides):
            itemsize = np.dtype(_array_dtype(array)).itemsize
            strides = tuple(int(s) // itemsize for s in array.strides)
        else:  # torch tensors: stride() is in elements
            strides = tuple(int(s) for s in array.stride())
        return Field.create_fixed_size(field_name, shape, index_dimensions, _array_dtype(array), strides=strides,
                                       field_type=field_type)

    _index_dimensions = 0

    # -- properties ----------------------------------------------------------------------------
    @property
    def dtype(self):
        return self._dtype

    @property
    def layout(self):
        return self._layout

    @property
    def index_dimensions(self):
        return self._index_dimensions

    @property
    def spatial_dimensions(self):
        return len(self.shape) - self._index_dimensions

    @property
    def spatial_shape(self) -> Tuple:
        return self.shape[:self.spatial_dimensions]

    @property
    def index_shape(self) -> Tuple:
        return self.shape[self.spatial_dimensions:]

    @property
    def spatial_strides(self):
        return self.strides[:self.spatial_dimensions]

    @property
    def has_fixed_shape(self):
        return all(isinstance(s, (int, np.integer)) for s in self.shape)

    @property
    def has_fixed_index_shape(self):
        return all(isinstance(s, (int, np.integer)) for s in self.index_shape)

    # -- accesses ------------------------------------------------------------------------------
    @property
    def center(self):
        return Field.Access(self, (0,) * self.spatial_dimensions)

    def __getitem__(self, offset):
        if isinstance(offset, np.ndarray):
            offset = tuple(offset)
        if isinstance(offset, str):
            raise NotImplementedError('direction-string offsets are not supported, pass integer tuples')
        if not isinstance(offset, (tuple, list)):
            offset = (offset,)
        offset = tuple(offset)
        if len(offset) != self.spatial_dimensions:
            raise ValueError('Wrong number of spatial indices: got %d, expected %d'
                             % (len(offset), self.spatial_dimensions))
        return Field.Access(self, offset)

    def __call__(self, *args, **kwargs):
        return self.center(*args, **kwargs)

    def neighbor(self, coord_id, offset):
        offs = [0] * self.spatial_dimensions
        offs[coord_id] = offset
        return Field.Access(self, tuple(offs))

    def new_field_with_different_name(self, new_name):
        f = Field(new_name, self.field_type, self._dtype, self._layout, self.shape, self.strides)
        f._index_dimensions = self._index_dimensions
        return f

    # -- identity ------------------------------------------------------------------------------
    def hashable_contents(self):
        return (self.name, self.field_type, self._dtype.numpy_dtype.str, self._index_dimensions,
                tuple(str(s) for s in self.shape))

    def __hash__(self):
        return hash(self.hashable_contents())

    def __eq__(self, other):
        return isinstance(other, Field) and self.hashable_contents() == other.hashable_contents()

    def __lt__(self, other):
        return self.name < other.name

    def __str__(self):
        return self.name

    def __repr__(self):
        return self.name

    # ------------------------------------------------------------------------------------------
    class Access(sp.Symbol):
        """Read/write of a field at a relative ``offsets`` (one per spatial dim) and ``index``."""

        def __new__(cls, field, offsets, index=()):
            offsets = tuple(_as_offset(o) for o in offsets)
            if not isinstance(index, (tuple, list)):
                index = (index,)
            index = tuple(int(i) if _is_intlike(i) else i for i in index)
            if all(isinstance(o, int) for o in offsets):
                offset_name = offset_to_direction_string(offsets)
            else:
                offset_name = '_'.join(str(o) for o in offsets)
            name = '%s_%s' % (field.name, offset_name)
            if index:
                name += '^' + '_'.join(str(i) for i in index)
            obj = sp.Symbol.__xnew__(cls, name)
            obj._field = field
            obj._offsets = offsets
            obj._index = index
            return obj

        def __getnewargs__(self):
            return self._field, self._offsets, self._index

        def __getnewargs_ex__(self):
            return (self._field, self._offsets, self._index), {}

        def __reduce_ex__(self, protocol):
            return Field.Access, (self._field, self._offsets, self._index)

        def _hashable_content(self):
            return (super()._hashable_content(), self._field.hashable_contents(),
                    tuple(str(o) for o in self._offsets), tuple(str(i) for i in self._index))

        def __call__(self, *idx):
            if not idx:
                return self
            if len(idx) == 1 and isinstance(idx[0], (tuple, list)):
                idx = tuple(idx[0])
            if self._index:
                raise ValueError('Indexing an already indexed Field.Access')
            if len(idx) != self._field.index_dimensions:
                raise ValueError('Wrong number of indices: got %d, expected %d'
                                 % (len(idx), self._field.index_dimensions))
            return Field.Access(self._field, self._offsets, idx)

        @property
        def field(self):
            return self._field

        @property
        def offsets(self):
            return self._offsets

        @property
        def index(self):
            return self._index

        @property
        def required_ghost_layers(self):
            return int(max([abs(int(o)) for o in self._offsets] + [0]))

        @property
        def is_absolute_access(self):
            return False

        @property
        def nr_of_coordinates(self):
            return len(self._offsets)

        def at_index(self, *idx):
            return Field.Access(self._field, self._offsets, idx)

        def get_shifted(self, *shift):
            return Field.Access(self._field, tuple(a + b for a, b in zip(shift, self._offsets)), self._index)

        def neighbor(self, coord_id, offset):
            offs = list(self._offsets)
            offs[coord_id] += offset
            return Field.Access(self._field, tuple(offs), self._index)

        def field_str(self):
            n = self._field.latex_name if self._field.latex_name else self._field.name
            offset_str = ','.join(str(o) for o in self._offsets)
            if self._index and self._index != (0,):
                return '%s[%s](%s)' % (n, offset_str, self._index if len(self._index) > 1 else self._index[0])
            return '%s[%s]' % (n, offset_str)

        def __format__(self, spec):
            return format(self.field_str(), spec)


def _is_intlike(v):
    return isinstance(v, (int, np.integer)) or (isinstance(v, sp.Basic) and v.is_Integer)


def _as_offset(o):
    if _is_intlike(o):
        return int(o)
    return sp.sympify(o)


def _array_dtype(array):
    dt = array.dtype
    if isinstance(dt, np.dtype):
        return dt
    return numpy_dtype_of_torch(dt)


def numpy_dtype_of_torch(dtype):
    """numpy dtype of a torch dtype: ``torch.bfloat16`` -> ``BFLOAT16``, the others by name."""
    name = str(dtype).replace('torch.', '')
    return BFLOAT16 if name == 'bfloat16' else np.dtype(name)


# ---------------------------------------------------------------------------------------------
_DESCR = re.compile(r'^\s*(?P<names>[^:]*?)\s*(?::\s*(?P<dtype>[A-Za-z_][A-Za-z0-9_]*)?\s*'
                    r'(?:\[(?P<size>[^\]]*)\])?)?\s*$')
_NAME_IDX = re.compile(r'\s*([A-Za-z_][A-Za-z0-9_]*)\s*(?:\(([^)]*)\))?\s*,?')


def _parse_description(description):
    m = _DESCR.match(description)
    if m is None:
        raise ValueError('Could not parse field description %r' % description)
    names_part = m.group('names')
    infos = []
    pos = 0
    while pos < len(names_part):
        mm = _NAME_IDX.match(names_part, pos)
        if mm is None or mm.end() == pos:
            raise ValueError('Could not parse field names in %r' % description)
        idx = tuple(int(i) for i in mm.group(2).split(',')) if mm.group(2) else ()
        infos.append((mm.group(1), idx))
        pos = mm.end()
    dtype = m.group('dtype') or 'float64'
    if dtype not in _C_TYPE_NAMES:
        raise ValueError('Unknown data type %r in field description' % dtype)
    size = m.group('size')
    if size is None:
        size_info = None
    else:
        size = size.strip()
        dm = re.match(r'^(\d+)\s*[dD]$', size)
        if dm:
            size_info = int(dm.group(1))  # symbolic shape with that many dims
        else:
            size_info = tuple(int(s) for s in size.split(',') if s.strip())
    return infos, np.dtype(_C_TYPE_NAMES[dtype]), size_info


def fields(description=None, index_dimensions=0, layout=None, field_type=FieldType.GENERIC, **kwargs):
    """``fields("z, y, x: float32[20,30]")`` / ``fields("a,b: [2D]")`` / ``fields(x=array)``.

    Mirrors the call sites in the reference (``pystencils.fields``): README.rst:55,
    tests/test_tfmad.py:191 (``"a, b, out: float64[5,7]"``), tests/test_autodiff.py:10
    (``"z, y, x: [2d]"``), tests/backends/test_torch_native_compilation.py:250 (``fields(x=tensor)``).
    """
    result = []
    if description:
        infos, dtype, size_info = _parse_description(description)
        for name, idx_shape in infos:
            if isinstance(size_info, tuple):
                f = Field.create_fixed_size(name, tuple(size_info) + tuple(idx_shape),
                                            index_dimensions=len(idx_shape), dtype=dtype, field_type=field_type)
            else:
                if size_info is None:
                    raise ValueError('Field description needs a size: "[20,30]" or "[2D]"')
                f = Field.create_generic(name, size_info, dtype=dtype, index_dimensions=len(idx_shape),
                                         index_shape=idx_shape, field_type=field_type)
            result.append(f)
    for name, arr in kwargs.items():
        result.append(Field.create_from_numpy_array(name, arr, index_dimensions=index_dimensions,
                                                    field_type=field_type))
    if len(result) == 0:
        return None
    if len(result) == 1:
        return result[0]
    return result


# ---------------------------------------------------------------------------------------------
# duck-typed import of foreign (real pystencils) objects
def coerce_field(f):
    if isinstance(f, Field):
        return f
    dtype = f.dtype.numpy_dtype if hasattr(f.dtype, 'numpy_dtype') else f.dtype
    out = Field(f.name, getattr(f, 'field_type', FieldType.GENERIC), dtype,
                tuple(range(f.spatial_dimensions)), tuple(f.shape), None)
    out._index_dimensions = f.index_dimensions
    out.latex_name = getattr(f, 'latex_name', None)
    return out


def coerce_access(a):
    if isinstance(a, Field.Access):
        return a
    return Field.Access(coerce_field(a.field), tuple(a.offsets), tuple(a.index))
