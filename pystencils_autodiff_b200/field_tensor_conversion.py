"""Tensor <-> Field front door (SURVEY.md §8 f-2).

Mirrors the conveniences of /root/reference/src/pystencils_autodiff/field_tensor_conversion.py:13-137 and
_backport.py:32-42 that users of the torch_native op touch: ``fields(x=tensor)``, ``create_field_from_array_like``,
``coerce_to_field``, ``is_array_like``, ``torch_tensor_from_field``.
"""
import numpy as np

from .field import Field, FieldType, fields  # noqa: F401  (fields(x=tensor) is the _backport.py:32-42 shim)

__all__ = ['ArrayWrapper', 'create_field_from_array_like', 'coerce_to_field', 'is_array_like',
           'torch_tensor_from_field', 'fields']


class ArrayWrapper:
    """Wraps an array/tensor and remembers index dimensions and field type (reference :13-42)."""

    def __init__(self, array, index_dimensions=0, field_type=FieldType.GENERIC, coordinate_transform=None,
                 spacing=None, origin=None):
        self.array = array
        self.index_dimensions = index_dimensions
        self.field_type = field_type
        self.coordinate_transform = coordinate_transform
        self.spacing = spacing
        self.origin = origin

    def __array__(self):
        return np.asarray(self.array)

    def __getattr__(self, name):
        return getattr(self.array, name)


def is_array_like(a):
    """numpy arrays, torch tensors and anything with ``shape`` + ``dtype`` (reference :97-105)."""
    import sympy as sp
    return (hasattr(a, '__array__') or (hasattr(a, 'shape') and hasattr(a, 'dtype'))) \
        and not isinstance(a, (sp.Matrix, sp.Basic, Field))


def create_field_from_array_like(field_name, maybe_array, annotations=None):
    """Field with the array's shape, strides and dtype (reference :55-88)."""
    index_dimensions, field_type = 0, FieldType.GENERIC
    if isinstance(maybe_array, ArrayWrapper):
        index_dimensions, field_type = maybe_array.index_dimensions, maybe_array.field_type
        maybe_array = maybe_array.array
    if annotations and isinstance(annotations, dict):
        index_dimensions = annotations.get('index_dimensions', index_dimensions)
        field_type = annotations.get('field_type', field_type)
    return Field.create_from_numpy_array(field_name, maybe_array, index_dimensions=index_dimensions,
                                         field_type=field_type)


def coerce_to_field(field_name, array_like):
    if is_array_like(array_like):
        return create_field_from_array_like(field_name, array_like)
    return array_like


def torch_tensor_from_field(field, init_val=0, cuda=True, requires_grad=False):
    """Tensor with the field's fixed shape and dtype (reference :132-137); CUDA by default."""
    import torch
    from .backends._torch_native import numpy_dtype_to_torch
    if not field.has_fixed_shape:
        raise ValueError('field %s has no fixed shape' % field.name)
    dtype = numpy_dtype_to_torch(field.dtype.numpy_dtype)
    shape = tuple(int(s) for s in field.shape)
    dev = 'cuda' if cuda else 'cpu'
    if init_val in (0, 0.0, False, None):
        t = torch.zeros(shape, dtype=dtype, device=dev)
    else:
        t = torch.full(shape, init_val, dtype=dtype, device=dev)
    return t.requires_grad_(requires_grad)
