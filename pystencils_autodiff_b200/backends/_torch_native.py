"""``torch_native`` backend: forward + adjoint stencil kernels as a ``torch.autograd.Function``.

Drop-in for /root/reference/src/pystencils_autodiff/backends/_torch_native.py:10-142
(``create_autograd_function(autodiff_obj, use_cuda, op_name=None)``), with the same marshalling rules
(SURVEY.md Appendix A-4): positional inputs bind to ``forward_input_fields`` (sorted by name), outputs are a
tuple in ``forward_output_fields`` order, backward binds ``grad_outputs[i]`` to the i-th ``diff<out>`` field and
returns the ``diff<in>`` tensors.  Differences, all deliberate:

* the kernels are the NVRTC-specialised sm_100a kernels of this package, launched through the C ABI on
  **torch's current stream** (the reference launches on the legacy default stream, printer.py:102-106);
* outputs are ``torch.empty`` — the kernels write every cell including the zero border — instead of
  ``torch.zeros`` + kernel (reference :64,:108: an extra HBM write pass per output);
* only the tensors the adjoint kernel actually reads are saved for backward (the reference stashes every
  kwarg, :84), so linear stencils save nothing;
* the gradient tuple is aligned with the positional inputs (``None`` for constant fields) — the reference
  returns one tensor per backward output and breaks with ``constant_fields`` (SURVEY.md Appendix B-5);
* CUDA only: ``use_cuda=False`` raises; there is no CPU path.
"""
import hashlib
from collections import OrderedDict

import numpy as np

from ..emit import emit_generic, emit_march, march_ineligible_reason
from ..emit_chain import chain_ineligible_reason, emit_march_chain
from ..field import BFLOAT16, BasicType
from ..ir import StencilKernelIR, lift_to_3d, split_index_components
from .. import runtime

__all__ = ['create_autograd_function', 'create_unrolled_function', 'compile_kernel', 'CompiledKernel',
           'numpy_dtype_to_torch']


def numpy_dtype_to_torch(dtype):
    """dtype name mapping (reference: backends/_pytorch.py:95-97); ``'bfloat16'`` / ``BFLOAT16`` -> ``torch.bfloat16``."""
    import torch
    dt = BasicType(dtype).numpy_dtype
    return torch.bfloat16 if dt == BFLOAT16 else getattr(torch, dt.name)


def launch_schedule(steps, pairs):
    """Steps per launch for ``steps`` applications of a stencil: fused pairs and the odd last step, or single steps."""
    return [2] * (steps // 2) + [1] * (steps % 2) if pairs else [1] * steps


class CompiledKernel:
    """One lowered kernel, callable like the reference's ``call_<kernel>(**tensors, **scalars)`` wrapper
    (backends/astnodes.py:143-146): fields are passed by name, outputs are written in place."""

    def __init__(self, ir: StencilKernelIR, tuning=None):
        self.ir = ir
        self.function_name = ir.function_name
        self.tuning = tuning
        self._emitted = {}
        self._native = {}
        # fields with an index dimension reach the fast path as one scalar field per component (SoA layouts only)
        self._scalar_ir, self._components = split_index_components(ir)
        self._march_reason = march_ineligible_reason(self._scalar_ir)
        if self._march_reason is None:
            try:
                self._emitted['march'] = emit_march(self._scalar_ir, tuning, masked=True)
                self._emitted['march_nomask'] = emit_march(self._scalar_ir, tuning, masked=False)
            except ValueError as e:
                self._march_reason = str(e)
        self._emitted['generic'] = emit_generic(ir)
        self.fields = ir.all_fields
        self.scalars = [s.name for s in ir.scalars]
        self.last_variant = None
        self._torch_dtypes = None
        # repeated launches (time loops, autograd Functions on the same buffers): everything the checks below derive from
        # (variant request, range, tensor identity = pointer + shape + strides + dtype) is remembered, so a repeat costs
        # one dictionary lookup and the C call
        self._field_names = [f.name for f in self.fields]
        self._fast = {}

    # -- introspection ---------------------------------------------------------------------------------------
    @property
    def code(self):
        return '\n'.join(self._emitted[k].source for k in sorted(self._emitted))

    @property
    def variants(self):
        return sorted(v for v in self._emitted if v in ('march', 'generic', 'march_x2'))

    def emitted(self, variant):
        if variant in ('march_peer', 'march_nomask_peer') and variant not in self._emitted:
            if 'march' not in self._emitted or self._components:
                raise ValueError('%s: peer halos need the march kernel (%s)' % (self.function_name, self._march_reason))
            self._emitted[variant] = emit_march(self._scalar_ir, self.tuning, masked=(variant == 'march_peer'), peer=True)
        if variant == 'march_x2_peer' and variant not in self._emitted:
            reason = self.fused_steps_reason() or ('needs 3-D fields' if self.ir.ndim != 3 else None)
            if reason:
                raise ValueError('%s: two fused steps per launch are not available: %s' % (self.function_name, reason))
            self._emitted[variant] = emit_march_chain(self.ir, self.tuning_x2, peer=True)
        if variant == 'march_x2' and variant not in self._emitted:
            reason = self.fused_steps_reason()         # emits the pair when it can be built
            if reason:
                raise ValueError('%s: two fused steps per launch are not available: %s' % (self.function_name, reason))
        return self._emitted[variant]

    def _chain_ir(self):
        """The kernel the fused-step emitter sees: 2-D 'zeros' kernels are lifted to 3-D fields of one plane."""
        if self.ir.ndim == 2 and self.ir.boundary == 'zeros' and not self._components:
            return lift_to_3d(self.ir)
        return self.ir

    tuning_x2 = None   # MarchTuning of the fused-step kernel (None = emit_chain defaults); set before the first use

    def fused_steps_reason(self):
        """None when ``out = S(S(u))`` can run as one launch (emit_chain.py), else why not.  The answer is the emitter's:
        the pair is emitted here (and kept), so that a stencil whose pair the tiling cannot hold — an x reach wider than a
        thread's strip, a y halo taller than the tile, a staged box or ring too large — takes single steps wherever pairs
        are the default instead of failing at its first launch."""
        try:
            return self._fused_reason          # asked per launch / per run() by the data handling: computed once
        except AttributeError:
            pass
        if self._components:
            reason = 'index dimensions'
        else:
            reason = self._march_reason or chain_ineligible_reason(self._chain_ir(), self.tuning_x2)
        if reason is None:
            try:
                self._emitted['march_x2'] = emit_march_chain(self._chain_ir(), self.tuning_x2)
            except ValueError as e:
                reason = str(e)
        self._fused_reason = reason
        return reason

    def run_steps(self, src, steps, out=None, fuse=None, **scalars):
        """``S^steps(src)``: the stencil applied ``steps`` times, ping-ponging between ``out`` and one scratch tensor;
        ``src`` is not modified.  ``fuse``: run pairs of steps as one launch (one read and one write of the field per
        pair instead of two).  Default: wherever a fused pair can be built (one-field stencils on dense aligned rows, 3-D
        or 2-D with the 'zeros' boundary) — measured wins on B200: 7-point fp32 at 1024^3 1.62x, 5-point fp32 at 8192^2
        1.39x, 27-point fp64 at 768^3 1.11x (two CTAs per SM, rows exchanged through shared memory)."""
        import torch
        if len(self.ir.input_fields) != 1 or len(self.ir.output_fields) != 1:
            raise ValueError('%s: run_steps needs a kernel with one input and one output field' % self.function_name)
        if steps < 1:
            raise ValueError('steps must be >= 1')
        fin, fout = self.ir.input_fields[0].name, self.ir.output_fields[0].name
        can_pair = self.fused_steps_reason() is None and self._select_variant([src, src]) == 'march'
        if fuse and not can_pair:
            raise ValueError('%s: steps cannot be fused: %s' % (self.function_name, self.fused_steps_reason() or
                                                                'tensor layout needs the generic kernel'))
        # pairs wherever they can be built: every measured case wins (round 2, scripts/steps_bench.py: 7-point fp32 1024^3
        # 1.62x, 5-point fp32 8192^2 — lifted to a one-plane 3-D field — 1.39x, 27-point fp64 768^3 1.11x)
        launches = launch_schedule(steps, can_pair if fuse is None else fuse)
        out = torch.empty_like(src) if out is None else out
        if out.data_ptr() == src.data_ptr():
            raise ValueError('%s: run_steps cannot work in place (out is src)' % self.function_name)
        scratch = torch.empty_like(src) if len(launches) > 1 else None
        cur = src
        for i, n in enumerate(launches):
            dst = out if (len(launches) - 1 - i) % 2 == 0 else scratch
            self(**{fin: cur, fout: dst}, _variant='march_x2' if n == 2 else None, **scalars)
            cur = dst
        return out

    def get_parameters(self):
        return self.ir.get_parameters()

    def native(self, variant, device_index=None):
        """``psad_kernel_t`` of a variant for one device (modules are loaded per CUDA context); must be called with
        that device current."""
        if device_index is None:
            import torch
            device_index = torch.cuda.current_device()
        key = (variant, device_index)
        if key not in self._native:
            self._native[key] = runtime.NativeKernel(self._emitted[variant])
        return self._native[key]

    def precompile(self):
        """NVRTC-compile every variant into the cubin cache (no GPU needed)."""
        logs = {}
        for v, ek in self._emitted.items():
            logs[v] = runtime.compile_source(ek.source, ek.cache_key, list(ek.options) + ['--ptxas-options=-v'])
        return logs

    # -- launch --------------------------------------------------------------------------------------------------
    def _select_variant(self, tensors):
        if 'march' not in self._emitted:
            return 'generic'
        nd = self.ir.ndim
        for f, t in zip(self.fields, tensors):
            es = t.element_size()
            # x (the last SPATIAL dim) must be contiguous; every other pitch — including the index dimension's for
            # structure-of-arrays vector fields — a multiple of 16 bytes
            if t.stride(nd - 1) != 1 or t.data_ptr() % 16 or (t.shape[nd - 1] * es) % 16:
                return 'generic'
            for d in range(t.dim()):
                if d != nd - 1 and (t.stride(d) * es) % 16:
                    return 'generic'
        return 'march'

    max_remembered_launches = 64

    def __call__(self, *, _range=None, _variant=None, _stream=None, _peer=None, **kwargs):
        """``_peer``: a ``runtime.Peer`` struct (neighbouring GPUs' arrays per field in plan order, completion counters,
        ``expect`` set by the caller) — the launch then uses the peer-halo instance of the march kernel."""
        try:
            key = [_variant, id(_range), id(_peer)]
            for n in self._field_names:
                t = kwargs[n]
                key += (t.data_ptr(), t.shape, t.stride(), t.dtype, t.is_cuda)
            hit = self._fast.get(tuple(key))
        except (KeyError, AttributeError, RuntimeError):
            hit = key = None        # missing / non-tensor argument: the checks below say what is wrong
        if hit is not None and hit[4] is _range and hit[8] is _peer:
            native, fa, n, dev_index, _, range_ref, self.last_variant, self.last_instance, _ = hit
            if _stream is None:
                _stream = _raw_current_stream(dev_index)
            native.launch_packed(fa, n, [float(kwargs[s]) for s in self.scalars] if self.scalars else (), _stream, range_ref,
                                 _peer)
            return None
        import torch
        if self._torch_dtypes is None:
            self._torch_dtypes = {f.name: numpy_dtype_to_torch(f.dtype.numpy_dtype) for f in self.fields}
        tensors = []
        for f in self.fields:
            if f.name not in kwargs:
                raise TypeError('%s: missing field argument %r' % (self.function_name, f.name))
            t = kwargs[f.name]
            if not isinstance(t, torch.Tensor) or not t.is_cuda:
                raise TypeError('%s: field %r must be a CUDA tensor (this backend has no CPU path)'
                                % (self.function_name, f.name))
            if t.dtype != self._torch_dtypes[f.name]:
                raise TypeError('%s: field %r expects dtype %s, got %s' % (self.function_name, f.name,
                                                                          f.dtype.numpy_dtype, t.dtype))
            if t.dim() != f.spatial_dimensions + f.index_dimensions:
                raise ValueError('%s: field %r expects %d dims, got shape %s'
                                 % (self.function_name, f.name, f.spatial_dimensions + f.index_dimensions, tuple(t.shape)))
            tensors.append(t)
        nd = self.ir.ndim
        shape0 = tuple(tensors[0].shape[:nd])
        dev = tensors[0].device
        for f, t in zip(self.fields, tensors):
            if tuple(t.shape[:nd]) != shape0:
                raise ValueError('%s: all fields must share one spatial shape: %r is %s, expected %s'
                                 % (self.function_name, f.name, tuple(t.shape[:nd]), shape0))
            if t.device != dev:
                raise ValueError('%s: all fields must live on the same device' % self.function_name)
        scal = []
        for s in self.scalars:
            if s not in kwargs:
                raise TypeError('%s: missing scalar argument %r' % (self.function_name, s))
            scal.append(float(kwargs[s]))
        variant = _variant or self._select_variant(tensors)
        if variant == 'march_x2':
            self.emitted(variant)
            if _range is not None and nd != 3:
                raise ValueError('%s: fused steps of 2-D kernels run on whole arrays only' % self.function_name)
            if self._select_variant(tensors) != 'march':
                raise ValueError('%s: fused steps need dense, 16-byte aligned rows' % self.function_name)
            if tensors[0].data_ptr() == tensors[1].data_ptr():
                raise ValueError('%s: input and output must be different tensors' % self.function_name)
        if variant == 'march':
            # the mask-free instance is valid whenever every written cell is also an evaluated cell
            if _range is not None:
                same = _range.get('_same')
                if same is None:
                    same = _range['_same'] = (list(_range['iter_lo'][:nd]) == list(_range['write_lo'][:nd]) and
                                              list(_range['iter_hi'][:nd]) == list(_range['write_hi'][:nd]))
            else:
                same = self.ir.boundary == 'zeros' or self.ir.ghost_layers == 0
            if same:
                variant = 'march_nomask'
        if _peer is not None:
            if not variant.startswith('march') or nd != 3:
                raise ValueError('%s: peer halos need the 3-D march kernel (this launch selected %r)'
                                 % (self.function_name, variant))
            variant += '_peer'
            self.emitted(variant)
        field_args = []
        if variant == 'march_x2' and nd == 2:
            # lifted kernel (lift_to_3d): the 2-D tensors are passed as one-plane 3-D fields
            for t in tensors:
                field_args.append((t.data_ptr(), (1,) + tuple(t.shape), [t.shape[0] * t.stride(0)] + list(t.stride()) + [0]))
        elif variant.startswith('march') and self._components:
            by_name = {f.name: t for f, t in zip(self.fields, tensors)}
            for cf in self._emitted['march'].fields:          # component fields, plan order of the scalar kernel
                name, i = self._components.get(cf.name, (cf.name, None))
                t = by_name[name]
                off = 0 if i is None else i * t.stride(nd) * t.element_size()
                if i is not None and i >= t.shape[nd]:
                    raise ValueError('%s: index %d out of range for field %r' % (self.function_name, i, name))
                field_args.append((t.data_ptr() + off, tuple(t.shape[:nd]), list(t.stride()[:nd]) + [0] * (4 - nd)))
        else:
            for f, t in zip(self.fields, tensors):
                st = list(t.stride()[:nd]) + [0] * (3 - nd)
                st.append(t.stride(nd) if f.index_dimensions else 0)
                field_args.append((t.data_ptr(), tuple(t.shape[:nd]), st))
        dev_index = dev.index if dev.index is not None else torch.cuda.current_device()
        with torch.cuda.device(dev):
            stream = _stream if _stream is not None else torch.cuda.current_stream(dev).cuda_stream
            native = self.native(variant, dev_index)
            if _peer is None:
                native.launch(field_args, scal, stream, _range)
            else:
                if _range is not None and '_ctypes' not in _range:
                    native.launch_range_struct(_range)
                import ctypes as _ct
                native.launch_packed(native.pack_fields(field_args), len(field_args), scal, stream,
                                     None if _range is None else _ct.byref(_range['_ctypes']), _peer)
        self.last_variant = 'march' if variant.startswith('march') else variant
        self.last_instance = variant
        # remember the validated launch (the range dict is held: its id() cannot be reused while the entry lives)
        if key is not None and (_range is None or '_ctypes' in _range):
            if len(self._fast) >= self.max_remembered_launches:
                self._fast.clear()
            range_ref = None
            if _range is not None:
                import ctypes
                range_ref = ctypes.byref(_range['_ctypes'])
            self._fast[tuple(key)] = (native, native.pack_fields(field_args), len(field_args), dev_index, _range, range_ref,
                                      self.last_variant, self.last_instance, _peer)
        return None


class _ShapeOnly:
    """Stand-in for a tensor where only ``.shape`` is needed."""

    def __init__(self, shape):
        self.shape = tuple(shape)


def _raw_current_stream(device_index):
    """``cudaStream_t`` of torch's current stream as an integer (the private fast accessor when it exists)."""
    import torch
    try:
        return torch._C._cuda_getCurrentRawStream(device_index)
    except AttributeError:
        return torch.cuda.current_stream(device_index).cuda_stream


_KERNEL_CACHE = {}


def compile_kernel(ir: StencilKernelIR, tuning=None) -> CompiledKernel:
    key = (id(ir), repr(tuning))
    if key not in _KERNEL_CACHE:
        _KERNEL_CACHE[key] = (ir, CompiledKernel(ir, tuning))
    return _KERNEL_CACHE[key][1]


def _hash(data):
    return hashlib.md5(data)


def create_autograd_function(autodiff_obj, use_cuda=True, op_name=None, tuning=None):
    import torch
    if not use_cuda:
        raise NotImplementedError('pystencils_autodiff_b200 is CUDA-only: use_cuda=False has no implementation')

    forward_ir = autodiff_obj.forward_ast_gpu
    backward_ir = autodiff_obj.backward_ast_gpu if autodiff_obj.backward_output_fields else None
    fwd_kernel = CompiledKernel(forward_ir, tuning)
    bwd_kernel = CompiledKernel(backward_ir, tuning) if backward_ir is not None else None

    if not op_name:
        digest = _hash((fwd_kernel.code + str(autodiff_obj) + str(autodiff_obj.constant_fields)).encode()).hexdigest()
        op_name = '%s_%s' % (autodiff_obj.op_name, digest)

    fwd_inputs = list(autodiff_obj.forward_input_fields)
    fwd_outputs = list(autodiff_obj.forward_output_fields)
    bwd_inputs = list(autodiff_obj.backward_input_fields)
    bwd_outputs = list(autodiff_obj.backward_output_fields)
    fwd_accessed = {f.name for f in forward_ir.fields_accessed}
    fwd_read = {f.name for f in forward_ir.fields_read}
    bwd_accessed = {f.name for f in backward_ir.fields_accessed} if backward_ir is not None else set()
    bwd_read = {f.name for f in backward_ir.fields_read} if backward_ir is not None else set()
    bwd_read_sorted = sorted(bwd_read)           # the order tensors are saved in must not depend on set iteration
    grad_fields = [f for f in bwd_inputs if f not in fwd_inputs and f not in fwd_outputs and f not in bwd_outputs]
    # which forward output each upstream-gradient field belongs to.  The reference binds ``grad_outputs[i]`` to the
    # i-th such field (:99-100), which is only right when the adjoint reads the gradient of EVERY output; here the
    # position comes from the forward output the adjoint field was derived from.
    grad_index = {}
    for i_, f in enumerate(grad_fields):
        fwd_f = getattr(f, 'corresponding_forward_field', None)
        names = [o.name for o in fwd_outputs]
        grad_index[f.name] = names.index(fwd_f.name) if fwd_f is not None and fwd_f.name in names else i_
    # adjoint of forward input i (None for constant fields)
    prefix_map = {}
    for f in bwd_outputs:
        fwd = getattr(f, 'corresponding_forward_field', None)
        prefix_map[fwd.name if fwd is not None else f.name] = f
    class_kwargs = dict()

    # per output field, once: fixed shape (or None), index shape, torch dtype — Function.apply / backward run per time step
    # and must not redo numpy dtype-name lookups or shape conversions (8 us each, measured)
    _alloc_info = {}
    for _f in list(fwd_outputs) + list(bwd_outputs):
        _alloc_info[_f.name] = (tuple(int(s_) for s_ in _f.shape) if _f.has_fixed_shape else None,
                                tuple(int(s_) for s_ in _f.index_shape), _f.spatial_dimensions,
                                numpy_dtype_to_torch(_f.dtype.numpy_dtype), bool(_f.index_dimensions))

    def _alloc(field, like, device, read_too):
        fixed, index_shape, nsp, dtype, has_index = _alloc_info[field.name]
        shape = fixed if fixed is not None else tuple(like.shape[:nsp]) + index_shape
        maker = torch.zeros if read_too else torch.empty
        if has_index:
            # vector outputs are allocated structure-of-arrays (x contiguous) so that they qualify for the fast path;
            # the returned tensor still has the field's logical shape [spatial..., index]
            t = maker(tuple(shape[nsp:]) + tuple(shape[:nsp]), dtype=dtype, device=device)
            return t.permute(*range(len(shape) - nsp, len(shape)), *range(len(shape) - nsp))
        return maker(shape, dtype=dtype, device=device)

    _grad_info = {f.name: (tuple(int(s_) for s_ in f.shape) if f.has_fixed_shape else None,
                           numpy_dtype_to_torch(f.dtype.numpy_dtype)) for f in grad_fields}
    fields_by_name = {f.name: f for f in list(fwd_inputs) + list(fwd_outputs) + list(bwd_inputs) + list(bwd_outputs)}

    def _device_layout(t, field=None):
        # the reference forces ``.cuda().contiguous()`` (:47-49).  Same here, except for vector fields that are stored
        # structure-of-arrays (x contiguous, dense): those keep their layout, it is the one the fast kernels want
        t = t.cuda()
        if field is not None and field.index_dimensions and t.dim() == field.spatial_dimensions + 1:
            nsp = field.spatial_dimensions
            if t.stride(nsp - 1) == 1:
                order = sorted(range(t.dim()), key=lambda d: -t.stride(d))
                if t.permute(*order).is_contiguous():
                    return t
            # array-of-structs (or strided) vector field: one transposing copy, then the fast kernels apply
            soa = t.permute(nsp, *range(nsp)).contiguous()
            return soa.permute(*range(1, nsp + 1), 0)
        return t if t.is_contiguous() else t.contiguous()

    def forward(ctx, *args, **kwargs):
        kwargs.update(class_kwargs)
        args = [_device_layout(a, fwd_inputs[i] if i < len(fwd_inputs) else None) if isinstance(a, torch.Tensor) else a
                for i, a in enumerate(args)]
        kwargs = {k: _device_layout(v, fields_by_name.get(k)) if isinstance(v, torch.Tensor) else v
                  for k, v in kwargs.items()}
        if len(args) > len(fwd_inputs):
            raise TypeError('%s takes %d input tensors (%s), got %d'
                            % (op_name, len(fwd_inputs), [f.name for f in fwd_inputs], len(args)))
        kwargs.update({f.name: args[i] for i, f in enumerate(fwd_inputs) if f.name in fwd_accessed and i < len(args)})
        first = next(v for v in list(args) + list(kwargs.values()) if isinstance(v, torch.Tensor))
        for f in fwd_outputs:
            if f.name not in kwargs:
                kwargs[f.name] = _alloc(f, first, first.device, f.name in fwd_read)
        outputs = OrderedDict((f.name, kwargs[f.name]) for f in fwd_outputs)
        fwd_kernel(**{k: v for k, v in kwargs.items() if k in fwd_accessed or k in fwd_kernel.scalars})
        # keep only what the adjoint kernel reads (tensors through save_for_backward, scalars on ctx)
        saved_names = [n for n in bwd_read_sorted if n in kwargs and isinstance(kwargs[n], torch.Tensor)]
        ctx.saved_names = saved_names
        ctx.save_for_backward(*[kwargs[n] for n in saved_names])
        ctx.saved_scalars = {k: v for k, v in kwargs.items() if not isinstance(v, torch.Tensor)}
        ctx.n_args = len(args)
        ctx.like = (first.shape, first.device)
        return tuple(outputs.values())

    def backward(ctx, *grad_outputs):
        if bwd_kernel is None:
            return tuple(None for _ in range(ctx.n_args))
        saved = dict(zip(ctx.saved_names, ctx.saved_tensors))
        shape, device = ctx.like
        gradients = {}
        for f in grad_fields:
            i = grad_index[f.name]
            g = grad_outputs[i] if i < len(grad_outputs) else None
            if g is None:
                g = torch.zeros(_grad_info[f.name][0] or shape, dtype=_grad_info[f.name][1], device=device)
            g = _device_layout(g, f) if g.is_cuda else g.contiguous()
            if not g.is_cuda:
                raise AssertionError('Some of the tensors where on the wrong device. Op was compiled for CUDA: True')
            if _grad_info[f.name][0] is not None and _grad_info[f.name][0] != tuple(g.shape):
                raise AssertionError('gradient for %s has shape %s, expected %s' % (f.name, tuple(g.shape), f.shape))
            gradients[f.name] = g
        # shape template for adjoint outputs of fields without a fixed shape: an upstream gradient, else a saved tensor,
        # else the forward call's first tensor (an adjoint with constant right-hand sides reads neither)
        like = next(iter(gradients.values())) if gradients else (next(iter(saved.values())) if saved else _ShapeOnly(shape))
        outs = OrderedDict((f.name, _alloc(f, like, device, f.name in bwd_read)) for f in bwd_outputs)
        kw = {**gradients, **saved, **outs}
        kw = {k: v for k, v in kw.items() if k in bwd_accessed}
        kw.update({k: v for k, v in ctx.saved_scalars.items() if k in bwd_kernel.scalars})
        bwd_kernel(**kw)
        result = []
        for i in range(ctx.n_args):
            adj = prefix_map.get(fwd_inputs[i].name)
            result.append(outs[adj.name] if adj is not None and adj.name in outs else None)
        return tuple(result)

    def call(cls, **kwargs):
        rtn = cls.apply(*[kwargs[p.symbol.name] for p in cls.forward_parameters])
        if len(rtn) == 1:
            rtn = rtn[0]
        return rtn

    cls = type(op_name, (torch.autograd.Function,), {
        'forward': staticmethod(forward),
        'backward': staticmethod(backward),
    })
    cls.class_kwargs = class_kwargs
    cls.kernel = staticmethod(forward)
    cls.ast = (fwd_kernel, bwd_kernel)
    cls.parameters = forward_ir.get_parameters()
    cls.forward_parameters = [p for p in cls.parameters if p.symbol.name in [f.name for f in fwd_inputs]]
    cls.forward_ast = forward_ir
    cls.backward_ast = backward_ir
    cls.forward_kernel = fwd_kernel
    cls.backward_kernel = bwd_kernel
    cls.num_regs = None
    cls.call = classmethod(call)
    cls.code = fwd_kernel.code + ('\n' + bwd_kernel.code if bwd_kernel is not None else '')
    return cls


def create_unrolled_function(autodiff_obj, steps, op_name=None, tuning=None, fuse=None):
    """``torch.autograd.Function`` for ``steps`` unrolled applications of a one-field stencil, ``u_T = S^T(u_0)``.

    The reference unrolls time steps by chaining ``op.apply`` calls (tests/test_tfmad.py style) — T forward and T
    adjoint launches, each a full read + write of the field, with T - 1 intermediate tensors kept alive by autograd.
    Here pairs of steps run as one launch (``CompiledKernel.run_steps``, emit_chain.py) and nothing is saved: the
    adjoint of a stencil whose adjoint kernel reads only the upstream gradient is ``(S^T)`` applied ``steps`` times to
    that gradient.  Stencils whose adjoint needs forward values are rejected (chain ``op.apply`` for those).
    ``fuse``: as in ``CompiledKernel.run_steps`` (None: pairs wherever they can be built; False: single steps — the
    results of a fused pair and of two single launches may differ in the last bit, the sums are ordered differently)."""
    import torch
    fwd_ir = autodiff_obj.forward_ast_gpu
    bwd_ir = autodiff_obj.backward_ast_gpu
    if len(fwd_ir.input_fields) != 1 or len(fwd_ir.output_fields) != 1:
        raise ValueError('unrolled steps need a stencil with one input and one output field')
    if len(bwd_ir.input_fields) != 1 or len(bwd_ir.output_fields) != 1:
        raise ValueError('unrolled steps need an adjoint that reads only the upstream gradient (a linear stencil)')
    if any(f.index_dimensions for f in fwd_ir.all_fields):
        raise ValueError('unrolled steps need scalar fields')
    steps = int(steps)
    fwd_kernel = CompiledKernel(fwd_ir, tuning)
    bwd_kernel = CompiledKernel(bwd_ir, tuning)
    dtype = numpy_dtype_to_torch(fwd_ir.input_fields[0].dtype.numpy_dtype)

    def _prep(t):
        t = t.cuda()
        if t.dtype != dtype:
            raise TypeError('expected a %s tensor, got %s' % (dtype, t.dtype))
        return t if t.is_contiguous() else t.contiguous()

    class_kwargs = dict()      # scalar parameters, like the single-step Function's class_kwargs

    def forward(ctx, u):
        ctx.scalars = dict(class_kwargs)
        return (fwd_kernel.run_steps(_prep(u), steps, fuse=fuse, **{k: v for k, v in ctx.scalars.items() if k in fwd_kernel.scalars}),)

    def backward(ctx, grad):
        return bwd_kernel.run_steps(_prep(grad), steps, fuse=fuse, **{k: v for k, v in ctx.scalars.items() if k in bwd_kernel.scalars})

    cls = type(op_name or '%s_x%d' % (autodiff_obj.op_name, steps), (torch.autograd.Function,),
               {'forward': staticmethod(forward), 'backward': staticmethod(backward)})
    cls.steps = steps
    cls.class_kwargs = class_kwargs
    cls.forward_kernel = fwd_kernel
    cls.backward_kernel = bwd_kernel
    cls.forward_ast = fwd_ir
    cls.backward_ast = bwd_ir
    return cls
