"""Slab-decomposed data handling with NCCL ghost-layer exchange (SURVEY.md §8e).

The reference has no distributed code: ``GraphDataHandling`` only *records* ``Communication(field, stencil, gpu)``
markers (/root/reference/src/pystencils_autodiff/graph_datahandling.py:87-91,305-316) while pystencils' serial
data handling does an in-process periodic copy, and ``PyTorchDataHandling.run_kernel`` simply calls the kernel with
all registered arrays (framework_integration/datahandling.py:185-188).  This module is where that marker becomes a
real exchange:

* every field is split along dim 0 (the slowest stride) into one slab per rank / GPU, stored with ``g`` ghost planes
  on each side — a ghost slab is one contiguous block, so faces are sent and received in place, no pack kernels;
* ``synchronization_function`` exchanges the boundary planes with the +-1 neighbours with grouped
  ``ncclSend``/``ncclRecv`` on a dedicated stream (C ABI: ``psad_halo_exchange``), or with ``torch.distributed``
  point-to-point ops (``backend='torch'``, which is what the CPU/gloo tests drive);
* kernels run on sub-ranges of the slab: interior planes while the halos are in flight, the ``g`` boundary planes
  on each side after the receive has completed (``cudaStreamWaitEvent``);
* because the adjoint is in gather form (TF-MAD) the backward pass needs the *same* exchange on ``diff<out>`` and
  nothing else — no reverse accumulation, no atomics.

Global boundary: ``'zeros'`` — the outermost ghost planes are never received and stay zero, which is exactly the
out-of-bounds-is-zero rule; ``None`` — the iteration range of the first / last rank is clipped to the global
interior.
"""
import ctypes
from collections import OrderedDict

import numpy as np

from . import runtime
from .backends._torch_native import CompiledKernel, launch_schedule, numpy_dtype_to_torch
from .field import BFLOAT16, BasicType, numpy_dtype_of_torch

__all__ = ['SlabDecomposition', 'HaloExchanger', 'SlabDataHandling', 'GraphDataHandling', 'PyTorchDataHandling',
           'create_slab_autograd_function', 'create_slab_unrolled_function',
           'SlabStencilOp', 'HostStreamedOp', 'TimeLoop']


import enum as _enum
import os as _os


def _host_array(t):
    """numpy copy of a tensor; bfloat16 is widened to float32 (exactly), numpy has no bfloat16."""
    import torch
    return (t.float() if t.dtype == torch.bfloat16 else t).cpu().numpy()


class SlabDecomposition:
    """Pure index logic of the 1-D decomposition along dim 0."""

    def __init__(self, global_shape, rank, world_size, ghost_layers, periodic=False):
        """``periodic``: the domain wraps around along dim 0 — the first and the last rank are neighbours (one rank: its own
        neighbour), the ghost planes at the global border receive the planes of the opposite end instead of staying zero."""
        self.global_shape = tuple(int(s) for s in global_shape)
        self.rank, self.world_size, self.g = int(rank), int(world_size), int(ghost_layers)
        self.periodic = bool(periodic)
        n0 = self.global_shape[0]
        base, rem = divmod(n0, world_size)
        self.counts = [base + (1 if r < rem else 0) for r in range(world_size)]
        self.starts = [sum(self.counts[:r]) for r in range(world_size)]
        self.n_local = self.counts[rank]
        self.start = self.starts[rank]
        if world_size > 1 and min(self.counts) < max(1, 2 * self.g):
            raise ValueError('slabs of %d planes are too thin for %d ghost layers' % (min(self.counts), self.g))

    @property
    def lo_rank(self):
        if self.periodic and self.world_size > 1:
            return (self.rank - 1) % self.world_size
        return self.rank - 1 if self.rank > 0 else -1

    @property
    def hi_rank(self):
        if self.periodic and self.world_size > 1:
            return (self.rank + 1) % self.world_size
        return self.rank + 1 if self.rank < self.world_size - 1 else -1

    @property
    def local_shape(self):
        """Shape of the local array including ghost planes."""
        return (self.n_local + 2 * self.g,) + self.global_shape[1:]

    @property
    def owned(self):
        return slice(self.g, self.g + self.n_local)

    def ranges(self, boundary, ghost_width_of_kernel, ndim, steps=1, halo=None):
        """(interior, lo, hi) launch ranges in local coordinates (``psad_range_t`` dicts); lo/hi may be None.

        ``boundary``: 'zeros' | 'none'; ``ghost_width_of_kernel``: iteration margin of the kernel in 'none' mode;
        ``steps`` > 1: ranges of a kernel that applies the stencil ``steps`` times per launch (``halo``: its reach along
        dim 0 per step)."""
        return slab_ranges(self.global_shape, self.start, self.n_local, self.g, self.lo_rank >= 0, self.hi_rank >= 0,
                           boundary, ghost_width_of_kernel, ndim, steps, halo, periodic=self.periodic)


def slab_ranges(global_shape, start, n, g, has_lo, has_hi, boundary, margin, ndim, steps=1, halo=None, periodic=False):
    """Launch ranges for the slab owning global planes ``[start, start+n)``, stored with ``g`` ghost planes.

    Returns ``(interior, lo, hi)``: the planes that do not depend on the ghost planes of a neighbour, and the planes
    next to each existing neighbour that do (None where there is none).  Cells inside ``[iter_lo, iter_hi)`` are
    evaluated, the other cells of ``[write_lo, write_hi)`` are set to 0 (``boundary='none'``: the global border).

    ``steps`` > 1 (kernels fusing several applications of a stencil that reaches ``halo`` planes along dim 0,
    emit_chain.py): a written plane depends on ``steps * halo`` planes on each side, so that many ghost planes must be
    stored (and exchanged once per launch instead of ``halo`` planes once per step), and that many planes next to a
    neighbour wait for the exchange.  The iteration range is then the part of the GLOBAL iteration space inside the local
    array — it also bounds the intermediate fields, which are needed (and valid) on ghost planes too."""
    shape = (n + 2 * g,) + tuple(global_shape[1:ndim])
    full_lo = [0] * ndim
    full_hi = list(shape)
    it_lo, it_hi = list(full_lo), list(full_hi)
    fused = steps > 1
    if fused:
        if halo is None or halo < 0:
            raise ValueError('fused steps: the reach of the stencil along dim 0 (halo) is required')
        if (has_lo or has_hi or periodic) and g < steps * halo:      # (one periodic rank is its own neighbour)
            raise ValueError('%d fused steps of a stencil reaching %d plane(s) need %d ghost planes, the slab stores %d'
                             % (steps, halo, steps * halo, g))
        if n < 2 * steps * halo and has_lo and has_hi:
            raise ValueError('slab of %d planes is too thin for %d fused steps' % (n, steps))
    if boundary == 'none' and margin > 0:
        for d in range(1, ndim):
            it_lo[d], it_hi[d] = margin, shape[d] - margin
        dom_lo, dom_hi = margin, global_shape[0] - margin
    else:
        dom_lo, dom_hi = 0, global_shape[0]
    if periodic:
        # no global border along dim 0: every plane the local array holds (ghost planes included) belongs to the domain
        dom_lo, dom_hi = start - g, start + n + g
    if fused:
        # global plane p lives at local index p - start + g
        it_lo[0] = max(dom_lo, start - g) - start + g
        it_hi[0] = max(it_lo[0], min(dom_hi, start + n + g) - start + g)
    elif boundary == 'none' and margin > 0:
        glo = max(dom_lo, start) - start + g
        ghi = min(dom_hi, start + n) - start + g
        it_lo[0], it_hi[0] = glo, max(glo, ghi)
    else:
        it_lo[0], it_hi[0] = g, g + n

    def rng(z0, z1):
        if z1 <= z0:
            return None
        if fused:
            return dict(iter_lo=list(it_lo), iter_hi=list(it_hi), write_lo=[z0] + full_lo[1:], write_hi=[z1] + full_hi[1:])
        lo = max(it_lo[0], z0)
        return dict(iter_lo=[lo] + it_lo[1:], iter_hi=[max(lo, min(it_hi[0], z1))] + it_hi[1:],
                    write_lo=[z0] + full_lo[1:], write_hi=[z1] + full_hi[1:])

    w = steps * halo if fused else g
    lo_w = min(w, n) if has_lo else 0
    hi_w = min(w, n - lo_w) if has_hi else 0
    if lo_w == 0 and hi_w == 0:
        return rng(g, g + n), None, None
    return rng(g + lo_w, g + n - hi_w), (rng(g, g + lo_w) if lo_w else None), (rng(g + n - hi_w, g + n) if hi_w else None)


def _reach(ir, name):
    """How many planes along dim 0 (the decomposed axis) ``ir`` reads field ``name`` away from the centre."""
    return max(ir.halo(name)[0])


def _exchanged_inputs(ir, dec):
    """Names of the input fields of ``ir`` whose ghost planes must be refreshed before a launch on ``dec``: ghost planes
    come from a neighbouring rank or, on a periodic domain, possibly from this rank's own far side."""
    if not (dec.world_size > 1 or dec.periodic) or dec.g == 0:
        return []
    return [f.name for f in ir.input_fields if _reach(ir, f.name) > 0]


def _fused_pair_reason(kernel, dec):
    """None when ``out = S(S(u))`` of ``kernel`` can run as one launch (``run_kernel(..., fused_steps=2)``) on ``dec``,
    else why not.  It is also the default wherever pairs are optional: every measured case wins (3-D 7-point fp32 1024^3
    per GPU: 1.63x / 1.71x at one / two GPUs; 27-point fp64 768^3: 1.08x / 1.07x, profiles/r2_slab_steps_c*_n*.json;
    2-D 5-point fp32 8192^2: 1.39x)."""
    ir = kernel.ir
    why = kernel.fused_steps_reason()
    if why is None and ir.ndim != 3:
        if dec.world_size > 1 or dec.g > 0:
            why = 'pairs of 2-D fields run on whole arrays only (one rank, no ghost planes)'
    elif why is None and (dec.world_size > 1 or dec.periodic):       # (one periodic rank is its own neighbour)
        need = 2 * _reach(ir, ir.input_fields[0].name)
        if dec.g < need:
            why = ('a pair needs %d ghost planes along dim 0 (twice the reach of the stencil), the data handling '
                   'stores %d ghost layers' % (need, dec.g))
    return None if why is None else '%s: steps cannot be fused: %s' % (kernel.function_name, why)


class HaloExchanger:
    """Neighbour exchange of ghost planes.  ``backend``: 'nccl' (C ABI, ``psad_halo_exchange``) or 'torch'
    (``torch.distributed`` P2P, any backend incl. gloo on CPU tensors)."""

    def __init__(self, decomposition, backend='nccl', group=None):
        self.dec = decomposition
        self.backend = backend
        self.group = group
        self._comm = None
        if decomposition.world_size > 1 and backend == 'nccl':
            self._init_nccl()

    def _init_nccl(self):
        import torch
        import torch.distributed as dist
        L = runtime.lib()
        buf = (ctypes.c_ubyte * 128)()
        if self.dec.rank == 0:
            runtime.check(L.psad_nccl_unique_id(buf), 'psad_nccl_unique_id')
        t = torch.tensor(list(buf), dtype=torch.uint8, device='cuda' if dist.get_backend(self.group) == 'nccl' else 'cpu')
        dist.broadcast(t, src=0, group=self.group)
        data = bytes(t.cpu().tolist())
        buf = (ctypes.c_ubyte * 128).from_buffer_copy(data)
        comm = ctypes.c_void_p()
        runtime.check(L.psad_nccl_comm_create(buf, self.dec.rank, self.dec.world_size, ctypes.byref(comm)),
                      'psad_nccl_comm_create')
        self._comm = comm

    def exchange(self, tensor, stream=None):
        """Fill the ghost planes of ``tensor`` (local array incl. ghosts, contiguous) from the neighbours."""
        dec = self.dec
        g, n = dec.g, dec.n_local
        if dec.world_size == 1 or g == 0:
            return
        self.exchange_planes(tensor[g:2 * g], tensor[0:g], tensor[n:n + g], tensor[n + g:n + 2 * g], stream)

    def exchange_planes(self, lo_send, lo_recv, hi_send, hi_recv, stream=None):
        """The exchange on explicitly given (contiguous, equally sized) blocks: ``lo_send`` goes to the lower neighbour,
        whose ``hi_send`` arrives in ``lo_recv``; likewise upwards.  Blocks towards a missing neighbour are ignored."""
        dec = self.dec
        if dec.world_size == 1:
            return
        if self.backend == 'nccl':
            nbytes = lo_send.numel() * lo_send.element_size()
            runtime.check(runtime.lib().psad_halo_exchange(
                self._comm, lo_send.data_ptr(), lo_recv.data_ptr(), hi_send.data_ptr(), hi_recv.data_ptr(),
                nbytes, dec.lo_rank, dec.hi_rank, ctypes.c_void_p(stream)), 'psad_halo_exchange')
        else:
            import torch.distributed as dist
            ops = []
            if dec.lo_rank >= 0 and dec.lo_rank == dec.hi_rank:
                # two ranks on a periodic domain: both neighbours are the same peer.  Messages between one pair of ranks
                # match in order, so the receives are posted in the order the peer sends: its first planes (our upper
                # ghost planes) first, its last planes (our lower ghost planes) second
                ops = [dist.P2POp(dist.isend, lo_send.contiguous(), dec.lo_rank, self.group),
                       dist.P2POp(dist.isend, hi_send.contiguous(), dec.hi_rank, self.group),
                       dist.P2POp(dist.irecv, hi_recv, dec.hi_rank, self.group),
                       dist.P2POp(dist.irecv, lo_recv, dec.lo_rank, self.group)]
            else:
                if dec.lo_rank >= 0:
                    ops.append(dist.P2POp(dist.isend, lo_send.contiguous(), dec.lo_rank, self.group))
                    ops.append(dist.P2POp(dist.irecv, lo_recv, dec.lo_rank, self.group))
                if dec.hi_rank >= 0:
                    ops.append(dist.P2POp(dist.isend, hi_send.contiguous(), dec.hi_rank, self.group))
                    ops.append(dist.P2POp(dist.irecv, hi_recv, dec.hi_rank, self.group))
            for req in dist.batch_isend_irecv(ops):
                req.wait()

    def close(self):
        if self._comm is not None:
            runtime.lib().psad_nccl_comm_destroy(self._comm)
            self._comm = None


class _PeerHalo:
    """Ghost planes read from the neighbouring GPUs' memory by the stencil kernel itself (``SlabDataHandling(peer_halo=True)``).

    The NCCL path runs, per kernel, an exchange of the boundary planes into the local ghost planes, one launch for the
    interior planes and one per side for the planes that had to wait.  Here every registered array is exported through CUDA
    IPC to the neighbouring ranks of the node, and ONE launch covers the whole slab: the kernel's producer warp stages
    the ghost planes by TMA straight from the neighbour's array over NVLink (``psad_kernel_launch_peer``, ``PSAD_PEER``
    in psad_march.cuh) — the halo transfer is part of the kernel's own pipeline, plane by plane, and nothing is copied
    twice.  Ordering between GPUs is a counter per rank in device memory: after its launch number k a rank stores k
    (stream order); launch k on a neighbour waits inside the kernel — only in the CTAs that touch ghost planes, and only
    before their first such load — until it reads k - 1 there.  That one condition covers both hazards (the neighbour has
    produced what is read, and has finished reading what is about to be overwritten) as long as all ranks issue the same
    sequence of launches, which an SPMD program does — and as long as the launch reaches at least as far along dim 0 as the
    launch before it did from the other side (the CTAs that overwrite planes a neighbour may still be reading are then CTAs
    that load ghost planes, hence wait).  A launch with a shorter reach, and every launch outside the protocol (kernels
    without a march instance, pointwise kernels), is preceded by ``psad_peer_wait``: a one-thread kernel that does the same
    wait in stream order.  Anything that changes an array outside the launch sequence (``fill``, ``to_gpu``, writes through
    ``owned()``) must be followed by ``fence()`` — ``fill`` / ``to_gpu`` do it themselves.  All launches of a data handling
    are expected on one stream (the counter is written in the order of the stream current at the launch).
    """

    def __init__(self, data_handling):
        import torch
        self.dh = data_handling
        self.torch = torch
        dec = data_handling.dec
        self.lo_rank, self.hi_rank = dec.lo_rank, dec.hi_rank
        self.seq = 0
        self.last_reach = (0, 0)         # planes the previous launch read below / above its own planes (from the neighbours)
        self.dirty = True                # arrays were written outside the launch sequence: fence before the next launch
        self.buffers = {}                # data_ptr of a registered array -> (lower neighbour's ptr, planes, upper ptr, planes)
        self.structs = {}
        self._keep = []
        self._opened = []
        self._ranges = {}
        # [0]: this rank's "launches completed" counter, [1]: error flag (a kernel gave up waiting for a neighbour)
        self.flags = torch.zeros(2, dtype=torch.int32, device=data_handling.device)
        (self.flag_lo, _), (self.flag_hi, _) = self._exchange(self.flags, 1)

    def _exchange(self, tensor, planes):
        """Collective: export ``tensor``, return ``((lower ptr, planes), (upper ptr, planes))`` of the neighbours' tensors
        registered in the same call (None where there is no neighbour)."""
        import torch.distributed as dist
        handle, offset = runtime.ipc_export(tensor.data_ptr())
        mine = (handle, offset, int(planes))
        everyone = [None] * self.dh.dec.world_size
        dist.all_gather_object(everyone, mine, group=self.dh.exchanger.group)
        out = []
        for r in (self.lo_rank, self.hi_rank):
            if r < 0:
                out.append((None, 0))
            else:
                h, off, pl = everyone[r]
                out.append((runtime.ipc_open(h, off), pl))
                self._opened.append(out[-1][0])
        self._keep.append(tensor)        # exported memory must stay alive while a neighbour maps it
        return out

    def register(self, tensor):
        (lo, lo_planes), (hi, hi_planes) = self._exchange(tensor, tensor.shape[0])
        self.buffers[tensor.data_ptr()] = (lo, lo_planes, hi, hi_planes)

    def close(self):
        """Collective: unmap the neighbours' arrays (they may be freed only after every rank that mapped them has closed
        them) and let go of the exported ones."""
        if self._opened is None:
            return
        import torch.distributed as dist
        self.fence()
        for p in self._opened:
            runtime.ipc_close(p)
        self._opened = None
        self.buffers.clear()
        self.structs.clear()
        dist.barrier(group=self.dh.exchanger.group)
        self._keep = []

    def applies(self, kernel, arrays, fused_steps):
        if kernel.ir.ndim != 3 or 'march' not in kernel._emitted or kernel._components:
            return False
        if any(t.data_ptr() not in self.buffers for t in arrays.values()):
            return False                 # an array that was not registered here (e.g. replaced by the user)
        return kernel._select_variant([arrays[f.name] for f in kernel.fields]) == 'march'

    def fence(self):
        """Every rank has finished everything it has launched: after this, arrays may be changed outside the launch
        sequence, and what was changed is visible to the neighbours' next launches."""
        import torch.distributed as dist
        self.torch.cuda.synchronize(self.dh.device)
        dist.barrier(group=self.dh.exchanger.group)
        self.dirty = False

    def errors(self):
        """1 if a kernel of this rank gave up waiting for a neighbour (host synchronisation)."""
        return int(self.flags[1].item())

    def _wait_in_stream(self):
        """The neighbours have finished their launch number ``seq`` (ours is about to be number ``seq + 1``)."""
        cur = self.torch.cuda.current_stream(self.dh.device).cuda_stream
        runtime.peer_wait(self.flag_lo, self.flag_hi, self.seq, self.flags.data_ptr() + 4, cur)

    def before_foreign_launch(self):
        """A launch outside the protocol is about to write arrays: the neighbours' previous launch may still be reading
        their boundary planes."""
        if self.dirty:
            self.fence()
        if self.last_reach != (0, 0):
            self._wait_in_stream()

    def count_foreign_launch(self):
        self.seq += 1
        self.last_reach = (0, 0)
        cur = self.torch.cuda.current_stream(self.dh.device).cuda_stream
        runtime.stream_write_u32(self.flags.data_ptr(), self.seq, cur)

    def run(self, kernel, arrays, fused_steps, kwargs):
        dh, dec = self.dh, self.dh.dec
        ir = kernel.ir
        if self.dirty:
            self.fence()
        key = (id(kernel), fused_steps)
        if key not in self._ranges:
            halo = _reach(ir, ir.input_fields[0].name) if fused_steps > 1 else None
            # ONE launch for all owned planes: nothing waits for an exchange
            whole = slab_ranges(dec.global_shape, dec.start, dec.n_local, dec.g, False, False, ir.boundary, ir.ghost_layers,
                                ir.ndim, fused_steps, halo, periodic=dec.periodic)[0]
            lo, hi = ir.max_halo[0]
            self._ranges[key] = (kernel, whole, (lo * fused_steps, hi * fused_steps))
        _, whole, reach = self._ranges[key]
        # the lower neighbour's previous launch read `last_reach[1]` of our lowest planes: the CTAs that overwrite them wait
        # for it if they load lower ghost planes, i.e. if this launch reaches as far down — likewise upwards
        if reach[0] < self.last_reach[1] or reach[1] < self.last_reach[0]:
            self._wait_in_stream()
        self.last_reach = reach
        tensors = [arrays[f.name] for f in kernel.fields]
        skey = (id(kernel),) + tuple(t.data_ptr() for t in tensors)
        peer = self.structs.get(skey)
        if peer is None:
            peer = runtime.Peer()
            for i, t in enumerate(tensors):
                lo, lo_planes, hi, hi_planes = self.buffers[t.data_ptr()]
                peer.lo_ptr[i], peer.hi_ptr[i] = lo, hi
                peer.lo_planes, peer.hi_planes = lo_planes or 0, hi_planes or 0
            peer.flag_lo, peer.flag_hi = self.flag_lo, self.flag_hi
            peer.error_flag = self.flags.data_ptr() + 4
            peer.ghost_planes = dec.g
            if len(self.structs) > 256:
                self.structs.clear()
            self.structs[skey] = peer
        self.seq += 1
        peer.expect = self.seq - 1
        kernel(**arrays, **kwargs, _range=whole, _peer=peer)
        runtime.stream_write_u32(self.flags.data_ptr(), self.seq, self.torch.cuda.current_stream(dh.device).cuda_stream)


PEER_HALO_MAX_CELLS = 600 * 1000 * 1000


def peer_halos_pay_off(local_shape, world_size, backend='nccl', device=None):
    """``peer_halo='auto'``: peer halos where they were measured to win (profiles/r2_peer_halo.md, two B200s over NVLink).
    One launch per kernel with the ghost planes read from the neighbours costs ~18 us per forward+adjoint step next to a GPU
    that has no neighbours at all, the NCCL exchange + interior / boundary launches 60-95 us — until the slabs get thick
    enough for the boundary launches to hide completely behind the interior one (7-point fp32, 1024 planes of 1024^2: NCCL
    +29 us, peer +54 us per step).  So: all ranks on one node, NCCL backend, 3-D slabs of at most 6e8 cells."""
    if world_size < 2 or backend != 'nccl' or len(local_shape) != 3:
        return False
    if device is not None and getattr(device, 'type', 'cuda') != 'cuda':
        return False
    local_world = _os.environ.get('LOCAL_WORLD_SIZE')
    if local_world is not None and int(local_world) != world_size:
        return False                     # ranks on several nodes: no peer memory between them
    if 'expandable_segments:True' in _os.environ.get('PYTORCH_CUDA_ALLOC_CONF', ''):
        return False                     # such allocations cannot be exported through CUDA IPC
    cells = 1
    for v in local_shape:
        cells *= int(v)
    return cells <= PEER_HALO_MAX_CELLS


class DataTransferKind(str, _enum.Enum):
    """Kinds of recorded data movement (graph_datahandling.py:21-38).  The queue entries of this data handling carry the
    member NAMES as strings (``('DataTransfer', name, 'HOST_TO_DEVICE')``): ``DataTransferKind(entry[2])`` gives the member."""
    UNKNOWN = 'UNKNOWN'
    HOST_ALLOC = 'HOST_ALLOC'
    DEVICE_ALLOC = 'DEVICE_ALLOC'
    HOST_TO_DEVICE = 'HOST_TO_DEVICE'
    DEVICE_TO_HOST = 'DEVICE_TO_HOST'
    HOST_COMMUNICATION = 'HOST_COMMUNICATION'
    DEVICE_COMMUNICATION = 'DEVICE_COMMUNICATION'
    HOST_SWAP = 'HOST_SWAP'
    DEVICE_SWAP = 'DEVICE_SWAP'
    HOST_GATHER = 'HOST_GATHER'
    DEVICE_GATHER = 'DEVICE_GATHER'

    def is_alloc(self):
        return self in (DataTransferKind.HOST_ALLOC, DataTransferKind.DEVICE_ALLOC)

    def is_transfer(self):
        # (the reference's version names a member that does not exist — ``self.SWAP`` — and raises; both swaps count here)
        return self in (DataTransferKind.HOST_TO_DEVICE, DataTransferKind.DEVICE_TO_HOST, DataTransferKind.HOST_SWAP,
                        DataTransferKind.DEVICE_SWAP)


class TorchArrayHandler:
    """``PyTorchDataHandling.PyTorchArrayHandler`` (framework_integration/datahandling.py:137-174): the array factory /
    transfer helper pystencils' serial data handling delegates to, on torch tensors.  Host arrays come from the factory
    methods, ``to_gpu`` / ``upload`` put them on the data handling's device."""

    def __init__(self, device=None):
        import torch
        self.torch = torch
        self.device = device
        self.from_numpy = torch.from_numpy

    def zeros(self, shape, dtype=np.float32, order='C'):
        assert order == 'C'
        return self.torch.zeros(*shape, dtype=numpy_dtype_to_torch(dtype))

    def ones(self, shape, dtype=np.float32, order='C'):
        assert order == 'C'
        return self.torch.ones(*shape, dtype=numpy_dtype_to_torch(dtype))

    def empty(self, shape, dtype=np.float32, layout=None):
        if layout not in (None, 'numpy', 'c', 'C') and tuple(layout) != tuple(range(len(shape))):
            raise NotImplementedError("only the 'numpy' (C order) layout is supported")
        return self.torch.empty(*shape, dtype=numpy_dtype_to_torch(dtype))

    def randn(self, shape, dtype=np.float32):
        return self.torch.randn(tuple(shape), dtype=numpy_dtype_to_torch(dtype))

    def _on_device(self, array):
        t = array if hasattr(array, 'cuda') else self.torch.from_numpy(array)
        return t.to(self.device) if self.device is not None else t.cuda()

    def to_gpu(self, array):
        return self._on_device(array)

    def upload(self, gpuarray, numpy_array):
        gpuarray[...] = self._on_device(numpy_array)

    def download(self, gpuarray, numpy_array):
        numpy_array[...] = gpuarray.cpu() if hasattr(numpy_array, 'cuda') else gpuarray.cpu().numpy()


class SlabDataHandling:
    """Array registry with the reference's data-handling vocabulary (``add_array``, ``fields``, ``run_kernel``,
    ``synchronization_function``, ``swap``, ``fill``, ``gather_array``; graph_datahandling.py:202-327,
    framework_integration/datahandling.py:54-200) on top of slab-decomposed CUDA tensors.  ``call_queue`` records
    what was executed with the reference's event names (``KernelCall``, ``Communication``, ``Swap``)."""

    def __init__(self, domain_size, rank=0, world_size=1, default_ghost_layers=1, device=None, backend='nccl',
                 group=None, periodic=False, peer_halo=False):
        """``periodic``: the domain is periodic along dim 0 (the decomposed axis): ghost-plane synchronisation wraps around
        — what pystencils' serial data handling does inside one array for the reference (graph_datahandling.py:305-316 →
        ``SerialDataHandling.synchronization_function``).  The other axes keep the kernels' own boundary treatment."""
        import torch
        self.torch = torch
        self.dec = SlabDecomposition(domain_size, rank, world_size, default_ghost_layers, periodic)
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device()) if torch.cuda.is_available() else torch.device('cpu')
        self.device = torch.device(device)
        self.exchanger = HaloExchanger(self.dec, backend, group)
        self.gpu_arrays = OrderedDict()
        self.cpu_arrays = OrderedDict()
        self.custom_data_cpu, self.custom_data_gpu, self._custom_data_transfer_functions = {}, {}, {}
        self.array_handler = TorchArrayHandler(self.device)
        self.fields = OrderedDict()
        self.call_queue = []
        self.kernel_io = {}            # kernel name -> (read field names, written field names) of the kernels run here
        self._swap_count = 0
        self._replicated = set()       # arrays with their own spatial shape: whole on every rank, no ghost planes
        self._range_cache = {}
        self._comm_stream = None
        self._ev_ready = None
        self._ev_halo = None
        # peer halos: the stencil kernels read their ghost planes from the neighbouring GPUs' arrays (CUDA IPC mappings,
        # NVLink) instead of having them exchanged first — see _PeerHalo
        # float16 and bfloat16 arrays always take the NCCL exchange: the peer-halo kernel instance is not built for them
        self._peer_forced = peer_halo is True
        if peer_halo == 'auto':
            peer_halo = peer_halos_pay_off(self.dec.local_shape, self.dec.world_size, backend, self.device)
        if peer_halo and periodic:
            raise ValueError('peer halos are not available on periodic domains (use the NCCL exchange)') if peer_halo is True else None
        self.peer = _PeerHalo(self) if (peer_halo and not periodic and self.dec.world_size > 1 and self.dec.g > 0) else None

    def close(self):
        """Collective when peer halos are on: unmaps the neighbours' arrays before anyone frees them."""
        if self.peer is not None:
            self.peer.close()
            self.peer = None

    max_recorded_calls = 1 << 16      # the reference records without bound; a long-running time loop must not leak

    def _record(self, entry):
        if len(self.call_queue) < self.max_recorded_calls:
            self.call_queue.append(entry)

    # -- arrays ------------------------------------------------------------------------------------------------
    @property
    def dim(self):
        return len(self.dec.global_shape)

    @property
    def shape(self):
        return self.dec.global_shape

    def add_array(self, name, values_per_cell=1, dtype=np.float32, spatial_shape=None, **_):
        """``spatial_shape``: an array of its own size (``MultiShapeDatahandling.add_array``,
        framework_integration/datahandling.py:73-132, "communication free applications"): stored whole on every rank,
        without ghost planes, never exchanged; kernels over such arrays run unsharded on every rank."""
        from .field import Field
        if name in self.gpu_arrays:
            raise ValueError('GPU Field with this name already exists')
        tail = () if values_per_cell in (1, (1,), ()) else (tuple(values_per_cell) if hasattr(values_per_cell, '__len__')
                                                              else (int(values_per_cell),))
        if spatial_shape is not None and tuple(int(v) for v in spatial_shape) != self.dec.global_shape:
            shape = tuple(int(v) for v in spatial_shape)
            self._replicated.add(name)
        else:
            shape = self.dec.local_shape
        dtype = BasicType(dtype).numpy_dtype
        arr = self.torch.zeros(shape + tail, dtype=numpy_dtype_to_torch(dtype), device=self.device)
        if self.peer is not None and dtype in (np.float16, BFLOAT16) and name not in self._replicated:
            if self._peer_forced:
                raise ValueError('peer halos are not available for %s arrays (peer_halo=False or \'auto\' exchange '
                                 'their ghost planes through NCCL)' % ('bfloat16' if dtype == BFLOAT16 else 'float16'))
            # 'auto': not registered, so every launch on this array takes the NCCL exchange (_PeerHalo.applies)
        elif self.peer is not None and name not in self._replicated:
            self.peer.register(arr)              # collective: every rank adds its arrays in the same order
        self.gpu_arrays[name] = arr
        self.fields[name] = Field.create_fixed_size(name, shape + tail, index_dimensions=len(tail), dtype=dtype)
        return self.fields[name]

    def add_arrays(self, description, dtype=np.float32, spatial_shape=None):
        """``"u, out"`` or the field-description syntax ``"x, y(2): float32[20,30]"`` (data type and per-array shape from
        the description, like ``MultiShapeDatahandling.add_arrays``, framework_integration/datahandling.py:54-71)."""
        if ':' in description:
            from .field import _parse_description
            infos, dt, size = _parse_description(description)
            shape = size if isinstance(size, tuple) and size else spatial_shape
            return tuple(self.add_array(n, values_per_cell=idx or 1, dtype=dt, spatial_shape=shape) for n, idx in infos)
        return tuple(self.add_array(n.strip(), dtype=dtype, spatial_shape=spatial_shape) for n in description.split(','))

    def add_custom_data(self, name, cpu_creation_function, gpu_creation_function=None, cpu_to_gpu_transfer_func=None,
                        gpu_to_cpu_transfer_func=None):
        """Data that is not a field array (graph_datahandling.py:272-277 records a marker and defers to pystencils' serial
        data handling): the creation functions are called once, their results kept under ``custom_data_cpu[name]`` /
        ``custom_data_gpu[name]``; with both transfer functions ``to_gpu(name)`` / ``to_cpu(name)`` call
        ``cpu_to_gpu_transfer_func(gpu_data, cpu_data)`` / ``gpu_to_cpu_transfer_func(gpu_data, cpu_data)``."""
        if (cpu_to_gpu_transfer_func is None) != (gpu_to_cpu_transfer_func is None):
            raise ValueError('For GPU data, both transfer functions have to be specified')
        if name in self.custom_data_cpu or name in self.gpu_arrays:
            raise ValueError('Data with this name has already been added')
        self._record(('CustomData', name))
        self.custom_data_cpu[name] = cpu_creation_function()
        if gpu_creation_function is not None:
            self.custom_data_gpu[name] = gpu_creation_function()
            if cpu_to_gpu_transfer_func is not None:
                self._custom_data_transfer_functions[name] = (cpu_to_gpu_transfer_func, gpu_to_cpu_transfer_func)

    def add_array_like(self, name, name_of_template_field):
        t = self.gpu_arrays[name_of_template_field]
        return self.add_array(name, dtype=numpy_dtype_of_torch(t.dtype))

    def fill(self, array_name, val, **_):
        self._record(('Fill', array_name))        # graph_datahandling.py:324-327 records 'Fill <name>'
        if self.peer is not None:
            self.peer.fence()                     # the neighbours may still be reading this array's boundary planes
        self.owned(array_name)[...] = val
        if self.peer is not None:
            self.peer.dirty = True

    def require_autograd(self, bool_val, *names):
        """framework_integration/datahandling.py:190-200 (which sets an attribute torch never reads — ``require_autograd``
        instead of ``requires_grad``); here the tensors really start / stop recording."""
        for n in names:
            for arrays in (self.cpu_arrays, self.gpu_arrays):
                if n in arrays:
                    arrays[n].requires_grad_(bool(bool_val))

    def extract_tensor(self, field, on_gpu=True, with_ghost_layers=False):
        """The registered tensor of a field (graph_datahandling.py:352-355 records a ``GhostTensorExtraction`` marker
        and returns nothing); ghost planes stripped unless asked for."""
        name = field if isinstance(field, str) else field.name
        self._record(('GhostTensorExtraction', name, bool(on_gpu), bool(with_ghost_layers)))
        t = (self.gpu_arrays if on_gpu else self.cpu_arrays)[name]
        return t if with_ghost_layers or name in self._replicated else t[self.dec.owned]

    def save_fields(self, fields, output_path, flag_field=None):
        """Records a ``FieldOutput`` marker like the reference (graph_datahandling.py:346-350) and writes this rank's
        owned planes to ``<output_path>.rank<r>.npz``.  bfloat16 arrays are written as float32 (an exact widening:
        numpy has no bfloat16)."""
        if isinstance(fields, str) or not hasattr(fields, '__iter__'):
            fields = [fields]
        names = [f if isinstance(f, str) else f.name for f in fields]
        self._record(('FieldOutput', tuple(names), output_path, flag_field))
        np.savez('%s.rank%d.npz' % (output_path, self.dec.rank),
                 **{n: _host_array(self.owned(n).detach()) for n in names})

    def merge_swaps_with_kernel_calls(self, call_queue=None):
        """A ``Swap`` recorded right after a ``KernelCall`` is folded into that call
        (graph_datahandling.py:329-344: the swap becomes the call's ``tmp_field_swaps``): the schedule a replayed graph
        needs is "kernel, then exchange roles of its buffers".  Returns the merged queue; ``call_queue`` defaults to
        (and then replaces) the recorded one.  Swaps here are pointer swaps and cost nothing either way."""
        own = call_queue is None
        queue = self.call_queue if own else call_queue
        merged = []
        for entry in queue:
            if (isinstance(entry, tuple) and entry[0] == 'Swap' and merged and isinstance(merged[-1], tuple)
                    and merged[-1][0] in ('KernelCall', 'KernelCall+Swap')):
                prev = merged[-1]
                swaps = prev[-1] if prev[0] == 'KernelCall+Swap' else ()
                body = prev[1:-1] if prev[0] == 'KernelCall+Swap' else prev[1:]
                pair = (entry[1], entry[2])
                merged[-1] = ('KernelCall+Swap',) + tuple(body) + (swaps + ((pair,) if pair not in swaps else ()),)
            else:
                merged.append(entry)
        if own:
            self.call_queue = merged
        return merged

    def __str__(self):
        return '\n'.join(str(c) for c in self.call_queue)

    def owned(self, name):
        return self.gpu_arrays[name] if name in self._replicated else self.gpu_arrays[name][self.dec.owned]

    # -- host mirrors (reference: GraphDataHandling.to_cpu / to_gpu record a DataTransfer, graph_datahandling.py:255-282)
    def to_cpu(self, name):
        if name in self._custom_data_transfer_functions:
            self._record(('CustomTransfer', name, 'DEVICE_TO_HOST'))       # graph_datahandling.py:279-282
            return self._custom_data_transfer_functions[name][1](self.custom_data_gpu[name], self.custom_data_cpu[name])
        self._record(('DataTransfer', name, 'DEVICE_TO_HOST'))
        self.cpu_arrays[name] = self.gpu_arrays[name].detach().to('cpu', copy=True)
        return self.cpu_arrays[name]

    def to_gpu(self, name):
        if name in self._custom_data_transfer_functions:
            self._record(('CustomTransfer', name, 'HOST_TO_DEVICE'))
            return self._custom_data_transfer_functions[name][0](self.custom_data_gpu[name], self.custom_data_cpu[name])
        self._record(('DataTransfer', name, 'HOST_TO_DEVICE'))
        if name not in self.cpu_arrays:
            raise KeyError('no host copy of %r: call to_cpu(%r) first or fill cpu_arrays[%r]' % (name, name, name))
        if self.peer is not None:
            self.peer.fence()
        self.gpu_arrays[name].copy_(self.cpu_arrays[name])
        if self.peer is not None:
            self.peer.dirty = True

    def all_to_cpu(self):
        for n in self.gpu_arrays:
            self.to_cpu(n)

    def all_to_gpu(self):
        for n in self.cpu_arrays:
            self.to_gpu(n)

    def swap(self, name1, name2, gpu=True):
        self._record(('Swap', name1, name2))
        self._swap_count += 1
        self.gpu_arrays[name1], self.gpu_arrays[name2] = self.gpu_arrays[name2], self.gpu_arrays[name1]

    def gather_array(self, name):
        """Global array on every rank (host numpy), ghost planes stripped.  A bfloat16 array is returned as float32 (an
        exact widening: numpy has no bfloat16)."""
        import torch.distributed as dist
        local = self.owned(name).contiguous()
        if self.dec.world_size == 1 or name in self._replicated:
            return _host_array(local)
        parts = [self.torch.empty((c,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
                 for c in self.dec.counts]
        dist.all_gather(parts, local) if len(set(self.dec.counts)) == 1 else self._all_gather_uneven(parts, local)
        return _host_array(self.torch.cat(parts, 0))

    def _all_gather_uneven(self, parts, local):
        import torch.distributed as dist
        for r in range(self.dec.world_size):
            if r == self.dec.rank:
                parts[r].copy_(local)
            dist.broadcast(parts[r], src=r)

    # -- communication ---------------------------------------------------------------------------------------------
    def _streams(self):
        if self._comm_stream is None:
            self._comm_stream = self.torch.cuda.Stream(device=self.device)
            self._ev_ready = self.torch.cuda.Event()
            self._ev_halo = self.torch.cuda.Event()
        return self._comm_stream

    def synchronization_function(self, names, stencil=None, target='gpu', **_):
        """Returns a callable that exchanges the ghost planes of ``names`` (reference: graph_datahandling.py:305-316
        records ``Communication(field, stencil, gpu)`` and then runs pystencils' serial copy)."""
        if isinstance(names, str):
            names = [names]

        def sync():
            for n in names:
                self._record(('Communication', n, stencil, target == 'gpu'))
                self.start_exchange(n)
            self.finish_exchange()
        return sync

    def start_exchange(self, name):
        """Asynchronous: exchange on the communication stream, ordered after everything already queued on the
        current stream."""
        if name in self._replicated:
            return False
        return self._start_exchange(self.gpu_arrays[name])

    def _start_exchange(self, t):
        """``start_exchange`` of the slab array ``t``; True where the communication stream was ordered behind the current
        one."""
        if self.dec.g == 0:
            return False
        if self.dec.world_size == 1:
            if self.dec.periodic:
                # one rank on a periodic domain is its own neighbour: two device copies on the current stream
                g, n = self.dec.g, self.dec.n_local
                t[:g].copy_(t[n:n + g])
                t[n + g:].copy_(t[g:2 * g])
            return False
        if t.is_cuda:
            comm = self._streams()
            cur = self.torch.cuda.current_stream(self.device)
            self._ev_ready.record(cur)
            comm.wait_event(self._ev_ready)
            if self.exchanger.backend == 'nccl':
                self.exchanger.exchange(t, comm.cuda_stream)
            else:
                with self.torch.cuda.stream(comm):
                    self.exchanger.exchange(t)
            self._ev_halo.record(comm)
            return True
        self.exchanger.exchange(t)
        return False

    def finish_exchange(self):
        """Make the current stream wait for the halos (device-side dependency only, no host sync)."""
        if self.dec.world_size == 1 or self.dec.g == 0 or self._comm_stream is None:
            return
        self.torch.cuda.current_stream(self.device).wait_event(self._ev_halo)

    def create_timeloop(self, use_cuda_graph=True, concurrent=True, fuse_steps=None):
        return TimeLoop(self, use_cuda_graph, concurrent, fuse_steps)

    # -- kernels ---------------------------------------------------------------------------------------------------
    def run_kernel(self, kernel, halo_fields=(), fused_steps=1, **kwargs):
        """``kernel(**arrays, **kwargs)`` on the owned planes.  ``halo_fields``: inputs whose ghost planes must be
        fresh.  Their exchange runs on the communication stream while the interior planes are computed on the
        current stream; the ``g`` boundary planes on each side are launched on the communication stream right behind
        the exchange, so they overlap with (and fill the tail of) the interior launch instead of serialising after it.
        The current stream then waits for that stream — a device-side dependency, no host synchronisation.

        ``fused_steps=2``: the kernel's two-steps-per-launch instance (emit_chain.py) — ``out = S(S(u))`` from ONE
        exchange of ``2 * halo`` ghost planes instead of two exchanges of ``halo`` planes; the data handling must store
        that many ghost layers."""
        if not isinstance(kernel, CompiledKernel):
            if isinstance(kernel, type) and isinstance(getattr(kernel, 'forward_kernel', None), CompiledKernel):
                # the Function class of op.create_tensorflow_op(backend='torch_native') (tests/test_datahandling.py:17-35
                # passes the op itself): its forward kernel on the registered arrays, outputs written in place
                return self.run_kernel(kernel.forward_kernel, halo_fields, fused_steps,
                                       **{**getattr(kernel, 'class_kwargs', {}), **kwargs})
            if callable(kernel) and self.dec.world_size == 1:
                # any other callable gets every registered array by name, like PyTorchDataHandling.run_kernel
                # (framework_integration/datahandling.py:185-188); it cannot be split into slab launches
                self._record(('KernelCall', getattr(kernel, '__name__', type(kernel).__name__)))
                return kernel(**{n: self.owned(n) for n in self.gpu_arrays}, **kwargs)
            raise TypeError('run_kernel expects a CompiledKernel (AutoDiffOp.forward_kernel_gpu / backward_kernel_gpu) or '
                            'the Function class of a torch_native op; arbitrary callables only on a single rank')
        if fused_steps not in (1, 2):
            raise ValueError('fused_steps must be 1 or 2')
        arrays = {f.name: self.gpu_arrays[f.name] for f in kernel.fields}
        replicated = [n for n in arrays if n in self._replicated]
        if not replicated:
            return self._launch(kernel, arrays, halo_fields, fused_steps, kwargs)
        self._record_launch(kernel, halo_fields, fused_steps)
        if len(replicated) != len(arrays):
            raise ValueError('%s mixes slab-decomposed arrays with arrays of their own shape (%s)'
                             % (kernel.function_name, ', '.join(sorted(replicated))))
        if fused_steps > 1:
            kwargs = dict(kwargs, _variant='march_x2')
        return kernel(**arrays, **kwargs)          # whole arrays, every rank, no exchange

    def _record_launch(self, kernel, halo_fields, fused_steps):
        for n in halo_fields:           # recorded in the reference's order: synchronisation, then the kernel call
            self._record(('Communication', n, None, True))
        self._record(('KernelCall', kernel.function_name) if fused_steps == 1 else
                     ('KernelCall', kernel.function_name, fused_steps))
        if kernel.function_name not in self.kernel_io:          # for computationgraph.ComputationGraph
            self.kernel_io[kernel.function_name] = ([f.name for f in kernel.ir.input_fields],
                                                    [f.name for f in kernel.ir.output_fields])

    def _launch(self, kernel, arrays, halo_fields, fused_steps, kwargs):
        """``run_kernel`` on the given slab arrays (field name -> tensor with ghost planes) instead of the registered
        ones."""
        self._record_launch(kernel, halo_fields, fused_steps)
        key = (id(kernel), fused_steps)
        if key not in self._range_cache:
            ir = kernel.ir
            if fused_steps == 1:
                ranges = self.dec.ranges(ir.boundary, ir.ghost_layers, ir.ndim)
            else:
                reason = _fused_pair_reason(kernel, self.dec)
                if reason:
                    raise ValueError(reason)
                # None for 2-D pairs: the arrays ARE the field (one rank, no ghost planes), the pair runs on them whole
                # like CompiledKernel.run_steps (lifted to a one-plane 3-D field by the emitter)
                ranges = None if ir.ndim != 3 else self.dec.ranges(ir.boundary, ir.ghost_layers, ir.ndim, fused_steps,
                                                                   _reach(ir, ir.input_fields[0].name))
            self._range_cache[key] = (kernel, ranges)      # holds the kernel: its id() cannot be reused while cached
        ranges = self._range_cache[key][1]
        if fused_steps > 1:
            kwargs = dict(kwargs, _variant='march_x2')
        if ranges is None:
            return kernel(**arrays, **kwargs)
        if self.peer is not None and self.peer.applies(kernel, arrays, fused_steps):
            return self.peer.run(kernel, arrays, fused_steps, kwargs)
        interior, lo, hi = ranges
        if self.peer is not None:
            self.peer.before_foreign_launch()     # the neighbours may still be reading what this launch overwrites
        ordered = [self._start_exchange(arrays[n]) for n in halo_fields]     # True where the comm stream waits for `cur`
        side = [r for r in (lo, hi) if r is not None]
        on_comm = bool(side) and self._comm_stream is not None and all(t.is_cuda for t in arrays.values())
        if on_comm:
            # the side launches read inputs produced on the current stream (and write outputs whose previous user may
            # still be pending there): order the communication stream behind it even when no exchange was started
            # in this call (start_exchange records the same dependency; a second record / wait is harmless)
            if not any(ordered):
                self._ev_ready.record(self.torch.cuda.current_stream(self.device))
                self._comm_stream.wait_event(self._ev_ready)
            for r in side:
                kernel(**arrays, **kwargs, _range=r, _stream=self._comm_stream.cuda_stream)
            self._ev_halo.record(self._comm_stream)
        if interior is not None:
            kernel(**arrays, **kwargs, _range=interior)
        if side and not on_comm:
            self.finish_exchange()
            for r in side:
                kernel(**arrays, **kwargs, _range=r)
        elif side or halo_fields:
            self.finish_exchange()
        if self.peer is not None:
            self.peer.count_foreign_launch()      # launches outside the peer protocol still advance the counters

    def run_steps(self, kernel, steps, fuse=None, **scalars):
        """``steps`` applications of a one-input / one-output stencil kernel as the reference's time loop runs them
        (graph_datahandling.py:152-194: kernel call, ghost-layer synchronisation, ``swap``): after every launch the
        input and output arrays are swapped, so the array registered under the INPUT field's name holds the current
        state when this returns and the one under the output field's name is scratch.

        ``fuse=True``: pairs of steps run as one launch with one exchange of ``2 * halo`` ghost planes
        (``run_kernel(..., fused_steps=2)``): per pair the field is read and written once instead of twice and one
        message per neighbour replaces two.  Needs ``default_ghost_layers >= 2 * halo``.  Default (``fuse=None``): pairs
        wherever they can run (``_fused_pair_reason``): 3-D fields on a data handling that stores enough ghost layers,
        2-D 'zeros' stencils on one rank without ghost planes; everything else runs single steps."""
        ir = kernel.ir
        if len(ir.input_fields) != 1 or len(ir.output_fields) != 1:
            raise ValueError('%s: run_steps needs a kernel with one input and one output field' % kernel.function_name)
        if steps < 0:
            raise ValueError('steps must be >= 0')
        fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
        halo = _exchanged_inputs(ir, self.dec)
        if fuse is None:
            fuse = _fused_pair_reason(kernel, self.dec) is None
        for n in launch_schedule(steps, fuse):
            self.run_kernel(kernel, halo_fields=halo, fused_steps=n, **scalars)
            self.swap(fin, fout)
        return self.gpu_arrays[fin]


class _SlabTensors:
    """Padded slab buffers of one data handling (``g`` ghost planes on each side of the ``n`` owned planes) for the slab
    autograd Functions: allocation, recognition of tensors that already are the owned part of such a buffer, and kernel
    launches on explicitly given buffers."""

    def __init__(self, data_handling):
        import weakref
        self.dh = data_handling
        self.g, self.n = data_handling.dec.g, data_handling.dec.n_local
        self.ours = weakref.WeakValueDictionary()    # id -> buffer allocated here: its ghost planes are ours to write

    def new_padded(self, dtype, like, zero):
        torch = self.dh.torch
        g, n = self.g, self.n
        t = (torch.zeros if zero else torch.empty)((n + 2 * g,) + tuple(like.shape[1:]), dtype=dtype, device=like.device)
        if not zero and g:
            t[:g].zero_()             # ghost planes at the global border are never received: they must read as 0
            t[g + n:].zero_()
        self.ours[id(t)] = t
        return t

    def padded_of(self, t, dtype, what):
        """The padded buffer ``t`` is the owned part of, else a fresh one holding a copy of ``t``."""
        g, n = self.g, self.n
        if t.shape[0] != n:
            raise ValueError('%s: expected this rank\'s %d owned planes, got shape %s' % (what, n, tuple(t.shape)))
        if t.dtype != dtype:
            raise TypeError('%s expects dtype %s, got %s' % (what, dtype, t.dtype))
        base = t._base
        if (base is not None and base.dim() == t.dim() and base.shape[0] == n + 2 * g and base.is_contiguous()
                and t.stride() == base.stride() and t.storage_offset() == base.storage_offset() + g * base.stride(0)
                and (self.ours.get(id(base)) is base or any(base is a for a in self.dh.gpu_arrays.values()))):
            return base
        p = self.new_padded(dtype, t, zero=False)
        p[g:g + n].copy_(t.detach())
        return p

    def owned(self, padded):
        return padded[self.g:self.g + self.n]

    def launch(self, kernel, arrays, halo, scalars, fused_steps=1):
        self.dh._launch(kernel, {f.name: arrays[f.name] for f in kernel.fields}, halo, fused_steps,
                        {k: v for k, v in scalars.items() if k in kernel.scalars})


def _slab_tensors(data_handling):
    if getattr(data_handling, '_slab_tensor_pool', None) is None:
        data_handling._slab_tensor_pool = _SlabTensors(data_handling)      # shared by every Function of this data handling
    return data_handling._slab_tensor_pool


def _check_scalars(kernels, scalars):
    for kern in kernels:
        missing = [s_ for s_ in kern.scalars if s_ not in scalars]
        if missing:
            raise TypeError('%s: missing scalar argument(s) %s' % (kern.function_name, missing))


def create_slab_autograd_function(op, data_handling, op_name=None, tuning=None, scalars=None, kernel_class=None):
    """``torch.autograd.Function`` of an ``AutoDiffOp`` on THIS RANK'S SLAB of slab-decomposed fields (SURVEY.md §8e): the
    sharded counterpart of ``op.create_tensorflow_op(backend='torch_native')`` with the same calling convention
    (backends/_torch_native.py:43-118 of the reference) — ``Op.apply(*inputs)`` takes the forward input fields in
    ``op.forward_input_fields`` order and returns a tuple in ``op.forward_output_fields`` order — where every tensor is
    the rank's OWNED planes ``[n_local, ...]`` of a field whose global extent along dim 0 is split over the ranks.

    forward: ghost planes of the inputs are exchanged with the neighbours (overlapped with the interior launch), the
    forward kernel runs on the owned planes.  backward: the SAME exchange on the upstream gradients ``diff<out>``, then
    the local adjoint kernel — the adjoint is in gather form, so there is no reverse exchange and nothing is accumulated
    across ranks.

    Slab tensors live inside padded buffers (``g`` ghost planes per side).  Outputs and gradients are returned as views
    of such buffers, and a tensor that already is such a view (an output of a slab Function of the same data handling,
    ``data_handling.owned(name)``) is used in place, so chained steps copy nothing; any other tensor is copied into a
    fresh padded buffer once.

    ``kernel_class``: the ``CompiledKernel`` subclass that launches (tests replay the emitted kernels on the CPU)."""
    import torch
    dh = data_handling
    dec = dh.dec
    g = dec.g
    pool = _slab_tensors(dh)
    KC = kernel_class or CompiledKernel
    fwd_ir, bwd_ir = op.forward_ast_gpu, op.backward_ast_gpu
    fwd_k, bwd_k = KC(fwd_ir, tuning), KC(bwd_ir, tuning)
    scalars = dict(scalars or {})
    _check_scalars((fwd_k, bwd_k), scalars)
    fwd_inputs, fwd_outputs = list(op.forward_input_fields), list(op.forward_output_fields)
    bwd_outputs = {f.name: f for f in op.backward_output_fields}
    fields = {f.name: f for f in list(op.forward_fields) + list(op.backward_fields)}
    # adjoint fields carry the forward field they belong to (AdjointField.corresponding_forward_field)
    grad_of, adjoint_of = {}, {}         # forward output -> upstream gradient field; forward input -> its gradient field
    for f in fields.values():
        fwd = getattr(f, 'corresponding_forward_field', None)
        if fwd is not None:
            (grad_of if fwd in fwd_outputs else adjoint_of)[fwd.name] = f.name
    sharded = dec.world_size > 1 or dec.periodic       # ghost planes are filled from a neighbour (possibly this rank)
    need = max([_reach(ir, f.name) for ir in (fwd_ir, bwd_ir) for f in ir.input_fields] + [0])
    if sharded and g < need:
        raise ValueError('the stencils reach %d plane(s) along dim 0, the data handling stores %d ghost layer(s)' % (need, g))
    fwd_halo = _exchanged_inputs(fwd_ir, dec)
    # the forward pass has refreshed the ghost planes of its inputs, and the backward pass reuses those buffers
    bwd_halo = [n for n in _exchanged_inputs(bwd_ir, dec) if n not in fwd_halo]
    fwd_reads = {f.name for f in fwd_ir.input_fields}
    bwd_reads = {f.name for f in bwd_ir.input_fields}

    def tdtype(f):
        return numpy_dtype_to_torch(f.dtype.numpy_dtype)

    def like_for(f, like):
        if not f.index_dimensions:
            return like
        return like.new_empty(tuple(like.shape[:len(dec.global_shape)]) + tuple(int(v) for v in f.index_shape))

    def forward(ctx, *inputs):
        if len(inputs) != len(fwd_inputs):
            raise TypeError('%s takes %d input tensors (%s), got %d' % (op.op_name, len(fwd_inputs),
                                                                         [f.name for f in fwd_inputs], len(inputs)))
        arrays = {f.name: pool.padded_of(t, tdtype(f), '%s: field %r' % (op.op_name, f.name))
                  for f, t in zip(fwd_inputs, inputs)}
        like = inputs[0]
        for f in fwd_outputs:
            arrays[f.name] = pool.new_padded(tdtype(f), like_for(f, like), zero=f.name in fwd_reads)
        pool.launch(fwd_k, arrays, fwd_halo, scalars)
        saved = [k for k in arrays if k in bwd_reads]
        ctx.saved_names = saved
        ctx.save_for_backward(*[arrays[k] for k in saved])
        ctx.like = like
        return tuple(pool.owned(arrays[f.name]) for f in fwd_outputs)

    def backward(ctx, *grad_outputs):
        arrays = dict(zip(ctx.saved_names, ctx.saved_tensors))
        like = ctx.like
        for f, go in zip(fwd_outputs, grad_outputs):
            name = grad_of.get(f.name)
            if name is None or name not in bwd_reads:
                continue
            gf = fields[name]
            if go is None:
                arrays[name] = pool.new_padded(tdtype(gf), like_for(gf, like), zero=True)
            else:
                arrays[name] = pool.padded_of(go if go.is_contiguous() else go.contiguous(), tdtype(gf),
                                              '%s: gradient %r' % (op.op_name, name))
        for name, f in bwd_outputs.items():
            arrays[name] = pool.new_padded(tdtype(f), like_for(f, like), zero=name in bwd_reads)
        pool.launch(bwd_k, arrays, bwd_halo, scalars)
        result = []
        for f in fwd_inputs:
            name = adjoint_of.get(f.name)
            result.append(pool.owned(arrays[name]) if name in bwd_outputs else None)
        return tuple(result)

    cls = type(op_name or op.op_name + '_slab', (torch.autograd.Function,),
               {'forward': staticmethod(forward), 'backward': staticmethod(backward)})
    cls.forward_kernel, cls.backward_kernel = fwd_k, bwd_k
    cls.forward_ast, cls.backward_ast = fwd_ir, bwd_ir
    cls.data_handling = dh
    cls.class_kwargs = scalars
    return cls


def create_slab_unrolled_function(op, data_handling, steps, fuse=None, op_name=None, tuning=None, scalars=None,
                                  kernel_class=None):
    """``steps`` unrolled applications of a one-field linear stencil on this rank's slab, ``u_T = S^T(u_0)``, as ONE
    autograd Function: the sharded counterpart of ``AutoDiffOp.create_unrolled_torch_op`` (backends/_torch_native.py:
    ``create_unrolled_function``).  forward = ``steps`` launches of the forward kernel with a ghost-plane exchange before
    each, ping-ponging between two padded buffers (the input is never written); backward = the adjoint kernel applied
    ``steps`` times to the upstream gradient the same way; nothing is saved.  ``fuse=True``: pairs of steps as one launch
    with ONE exchange of ``2 x reach`` ghost planes per pair (needs that many ghost layers); ``fuse=None``: pairs where they
    are a measured win and possible (see ``SlabDataHandling.run_steps``)."""
    import torch
    dh = data_handling
    dec = dh.dec
    pool = _slab_tensors(dh)
    KC = kernel_class or CompiledKernel
    fwd_ir, bwd_ir = op.forward_ast_gpu, op.backward_ast_gpu
    for ir, what in ((fwd_ir, 'a stencil with one input and one output field'),
                     (bwd_ir, 'an adjoint that reads only the upstream gradient (a linear stencil)')):
        if len(ir.input_fields) != 1 or len(ir.output_fields) != 1:
            raise ValueError('unrolled steps need ' + what)
    steps = int(steps)
    if steps < 1:
        raise ValueError('steps must be >= 1')
    fwd_k, bwd_k = KC(fwd_ir, tuning), KC(bwd_ir, tuning)
    scalars = dict(scalars or {})
    _check_scalars((fwd_k, bwd_k), scalars)
    sharded = dec.world_size > 1 or dec.periodic       # ghost planes are filled from a neighbour (possibly this rank)
    reason = _fused_pair_reason(fwd_k, dec) or _fused_pair_reason(bwd_k, dec)
    if fuse and reason:
        raise ValueError(reason)
    launches = launch_schedule(steps, reason is None if fuse is None else fuse)
    for kern in (fwd_k, bwd_k):
        ir = kern.ir
        reach = _reach(ir, ir.input_fields[0].name)
        if sharded and dec.g < reach:
            raise ValueError('%s reaches %d plane(s) along dim 0, the data handling stores %d ghost layers'
                             % (kern.function_name, reach, dec.g))
    halos = {k: _exchanged_inputs(k.ir, dec) for k in (fwd_k, bwd_k)}

    def run(kernel, t):
        ir = kernel.ir
        fin, fout = ir.input_fields[0], ir.output_fields[0]
        dtype = numpy_dtype_to_torch(fin.dtype.numpy_dtype)
        cur = pool.padded_of(t if t.is_contiguous() else t.contiguous(), dtype, '%s: field %r' % (op.op_name, fin.name))
        halo = halos[kernel]
        spare = [pool.new_padded(dtype, t, zero=False) for _ in range(min(2, len(launches)))]
        for i, k in enumerate(launches):
            dst = spare[i % len(spare)]
            pool.launch(kernel, {fin.name: cur, fout.name: dst}, halo, scalars, fused_steps=k)
            cur = dst
        return pool.owned(cur)

    def forward(ctx, u):
        return (run(fwd_k, u),)

    def backward(ctx, grad):
        return run(bwd_k, grad)

    cls = type(op_name or '%s_slab_x%d' % (op.op_name, steps), (torch.autograd.Function,),
               {'forward': staticmethod(forward), 'backward': staticmethod(backward)})
    cls.steps, cls.launches = steps, launches
    cls.forward_kernel, cls.backward_kernel = fwd_k, bwd_k
    cls.forward_ast, cls.backward_ast = fwd_ir, bwd_ir
    cls.data_handling = dh
    cls.class_kwargs = scalars
    return cls


class GraphDataHandling(SlabDataHandling):
    """``SlabDataHandling`` behind the reference's constructor (graph_datahandling.py:196-200 /
    framework_integration/datahandling.py:176-183: ``(domain_size, default_ghost_layers, default_layout, periodicity,
    default_target)``).  Rank and world size come from ``torch.distributed`` when a process group is initialised, so the
    same script runs on one GPU or slab-decomposed under torchrun.  ``periodicity``: ``False``, or periodic along dim 0 only
    (``(True, False, ...)``: the decomposed axis, where ghost planes exist; arrays carry no ghost cells along the other axes,
    so periodicity there raises); layouts other than 'numpy' (C order) raise; ``default_target`` must be 'gpu'."""

    def __init__(self, domain_size, default_ghost_layers=0, default_layout='numpy', periodicity=False,
                 default_target='gpu', device=None, backend=None):
        import torch.distributed as dist
        nd = len(domain_size)
        per = tuple(bool(p) for p in periodicity) if hasattr(periodicity, '__iter__') else (bool(periodicity),) * nd
        if any(per[1:]):
            raise NotImplementedError('periodicity is supported along dim 0 only (the decomposed axis, where ghost planes '
                                      'exist): pass periodicity=(True,%s)' % (' False,' * (nd - 1)))
        if default_layout not in ('numpy', 'c', 'C'):
            raise NotImplementedError("only the 'numpy' (C order) layout is supported")
        if default_target not in ('gpu', None):
            raise NotImplementedError("this backend has no CPU path: default_target must be 'gpu'")
        rank, world = (dist.get_rank(), dist.get_world_size()) if dist.is_available() and dist.is_initialized() else (0, 1)
        if backend is None:
            backend = 'nccl' if (world == 1 or dist.get_backend() == 'nccl') else 'torch'
        super().__init__(domain_size, rank, world, default_ghost_layers, device, backend, periodic=per[0])
        self.default_target = 'gpu'


PyTorchDataHandling = GraphDataHandling     # framework_integration/datahandling.py:135


class TimeLoop:
    """Recorded sequence of steps, replayed ``n`` times (SURVEY.md §8 f-1 / f-3).

    API of the reference's ``GraphDataHandling.TimeLoop`` (graph_datahandling.py:152-194: ``add_pre_run_function``,
    ``add_post_run_function``, ``add_single_step_function``, ``add_call``, ``run``).  On one GPU the body of a time step
    (kernel launches and swaps) is captured once into a **CUDA graph** and replayed, which removes the per-launch host
    latency for small fields; with more than one rank (halo exchange inside the step) the calls are issued eagerly.

    **Scheduling from the dependency graph** (f-3, the reference's ``ComputationGraph`` over a call queue,
    computationgraph.py:17-163): when every part of the step was added through ``add_call(kernel, ...)`` / ``swap`` the
    loop knows what each call reads and writes, derives the levels of mutually independent calls
    (``computationgraph.ComputationGraph.levels``) and — on one rank — issues the calls of one level on different streams,
    forked from and joined back into the current stream with events.  Inside the captured CUDA graph those become parallel
    branches.  ``levels()`` shows the schedule; ``concurrent=False`` turns it off.

    **Fused pairs of steps** (f-1): a loop whose step is ``add_call(kernel)`` + ``swap(input, output)`` of a one-field stencil
    runs two time steps per launch (``fused_pair``; ``fuse_steps=False`` turns it off, ``True`` insists), on one GPU and on
    slabs (one exchange of twice the reach per pair) — the reference's own loop idiom gets what ``run_steps`` does.
    """

    def __init__(self, data_handling, use_cuda_graph=True, concurrent=True, fuse_steps=None):
        self.dh = data_handling
        self.concurrent = concurrent
        self.fuse_steps = fuse_steps      # None: fused pairs where run_steps() would take them; False: never; True: must
        self._entries = []                # structured step parts: ('kernel', kernel, kwargs, halo) | ('swap', a, b) | None
        self._side_streams = []
        self._pre, self._post, self._steps = [], [], []
        self._single_step_asts = []       # what one step consists of, in the reference's vocabulary (for TimeloopRun)
        self.time_steps_run = 0
        self._graphs = {}                 # buffer roles at capture time -> CUDA graph of two steps
        self._step_record = None          # what the data handling recorded during one executed step
        self.use_cuda_graph = use_cuda_graph

    max_cached_graphs = 4
    fused_last_run = False            # whether the last run() issued fused pairs of steps
    capture_error = None              # why the last CUDA-graph capture failed (the loop then runs eagerly), else None

    @property
    def parent(self):                     # the reference's name for the data handling (graph_datahandling.py:155)
        return self.dh

    def add_pre_run_function(self, f):
        self._pre.append(f)

    def add_post_run_function(self, f):
        self._post.append(f)

    def add_single_step_function(self, f, _entry=None):
        self._steps.append(f)
        self._entries.append(_entry)      # None: an opaque function — the step is then issued in program order
        self._graphs.clear()
        self._step_record = None
        self._levels = None
        self._fused = None

    def add_call(self, functor, argument_list=None):
        args = argument_list if argument_list is not None else {}
        if isinstance(args, dict):
            args = [args]
        for a in args:
            if isinstance(functor, CompiledKernel):
                halo = a.pop('halo_fields', ()) if isinstance(a, dict) else ()
                self._single_step_asts.append(('KernelCall', functor.function_name))
                self.add_single_step_function(lambda k=functor, kw=a, h=halo: self.dh.run_kernel(k, halo_fields=h, **kw),
                                              _entry=('kernel', functor, a, tuple(halo)))
            else:
                self._single_step_asts.append(('Call', getattr(functor, '__name__', type(functor).__name__)))
                self.add_single_step_function(lambda f=functor, kw=a: f(**kw))

    def swap(self, src, dst, is_gpu=True):
        """graph_datahandling.py:192-197 appends a ``Swap`` to the step's record; here the step also performs it (the
        reference only records because its queue is compiled later — this data handling executes)."""
        src = src if isinstance(src, str) else src.name
        dst = dst if isinstance(dst, str) else dst.name
        self._single_step_asts.append(('Swap', src, dst))
        self.add_single_step_function(lambda a=src, b=dst: self.dh.swap(a, b, is_gpu), _entry=('swap', src, dst))

    _levels = None

    def levels(self):
        """The step as levels of mutually independent parts (lists of indices into the step's parts, in order), from the
        array versions each part reads and writes; None when the step contains an opaque function."""
        if self._levels is None:
            if not self._entries or any(e is None for e in self._entries):
                return None
            from .computationgraph import ComputationGraph
            queue, io = [], {}
            for e in self._entries:
                if e[0] == 'kernel':
                    k = e[1]
                    io[k.function_name] = ([f.name for f in k.ir.input_fields], [f.name for f in k.ir.output_fields])
                    queue.append(('KernelCall', k.function_name))
                else:
                    queue.append(('Swap', e[1], e[2]))
            graph = ComputationGraph(queue, io)
            self._levels = [[n.index for n in level] for level in graph.levels()]
        return self._levels

    def fused_pair(self):
        """``(kernel, scalars, halo_fields)`` when two steps of this loop can run as ONE launch, else None (SURVEY §8 f-1).

        The reference's time-loop idiom — ``add_call(kernel)`` then ``swap(in, out)`` (graph_datahandling.py:152-197, the
        pair ``merge_swaps_with_kernel_calls`` folds into one node, :329-344) — is recognised when the kernel is a
        one-field stencil whose pair can run on this data handling (``_fused_pair_reason``, the rule
        ``SlabDataHandling.run_steps`` fuses by), for the default ``fuse_steps=None`` and ``True`` alike.  ``run`` then
        issues ``out = S(S(u))`` + one swap per two time steps — one read and one write of the field, one halo exchange of
        twice the reach — exactly what ``run_steps`` does, through the reference's API.  Results can differ from single
        steps in the last bit (sums are ordered differently)."""
        if self.fuse_steps is False:
            return None
        if self._fused is None or self._fused[0] is not self.fuse_steps:
            # decided once per step definition and setting (add_single_step_function resets it)
            self._fused = (self.fuse_steps, self._find_fused_pair())
        return self._fused[1]

    _fused = None                             # (fuse_steps it was decided for, None | (kernel, scalars, halo_fields))

    def _find_fused_pair(self):
        e = self._entries
        ok = (len(e) == 2 and e[0] is not None and e[1] is not None and e[0][0] == 'kernel' and e[1][0] == 'swap')
        why = 'the step is not `add_call(kernel)` followed by `swap(input, output)`'
        if ok:
            kernel, kw, halo = e[0][1], e[0][2], e[0][3]
            ir = kernel.ir
            ok = len(ir.input_fields) == 1 and len(ir.output_fields) == 1
            why = 'the kernel is not a one-input / one-output stencil'
        if ok:
            fin, fout = ir.input_fields[0].name, ir.output_fields[0].name
            ok = {e[1][1], e[1][2]} == {fin, fout} and all(n == fin for n in halo) and \
                all(isinstance(v, (int, float)) and not isinstance(v, bool) for v in kw.values())
            why = 'the swap does not exchange the kernel\'s input and output arrays (or the call passes non-scalar arguments)'
        if ok:
            why = _fused_pair_reason(kernel, self.dh.dec)
            ok = why is None
        if not ok:
            if self.fuse_steps is True:
                raise ValueError('TimeLoop(fuse_steps=True): %s' % why)
            return None
        return kernel, dict(kw), tuple(_exchanged_inputs(ir, self.dh.dec))

    def _one_pair(self, fused):
        kernel, kw, halo = fused
        ir = kernel.ir
        self.dh.run_kernel(kernel, halo_fields=halo, fused_steps=2, **kw)
        self.dh.swap(ir.input_fields[0].name, ir.output_fields[0].name)

    def _one_step(self):
        n = len(self.dh.call_queue)
        levels = self.levels() if (self.concurrent and self.dh.dec.world_size == 1) else None
        torch = self.dh.torch
        if levels is None or all(len(lv) == 1 for lv in levels) or not torch.cuda.is_available() \
                or not all(t.is_cuda for t in self.dh.gpu_arrays.values()):
            for f in self._steps:
                f()
        else:
            cur = torch.cuda.current_stream(self.dh.device)
            for lv in levels:
                kernels = [i for i in lv if self._entries[i][0] == 'kernel']
                if len(kernels) > 1:
                    while len(self._side_streams) < len(kernels) - 1:
                        self._side_streams.append(torch.cuda.Stream(self.dh.device))
                    fork = torch.cuda.Event()
                    fork.record(cur)
                    self._steps[kernels[0]]()
                    for s_, i in zip(self._side_streams, kernels[1:]):
                        s_.wait_event(fork)
                        with torch.cuda.stream(s_):
                            self._steps[i]()
                        cur.wait_stream(s_)
                else:
                    for i in kernels:
                        self._steps[i]()
                for i in lv:                       # swaps are host-side role changes: in order, after the level's launches
                    if self._entries[i][0] != 'kernel':
                        self._steps[i]()
        if self._step_record is None:
            self._step_record = tuple(self.dh.call_queue[n:])

    def _roles(self):
        """Identity of every registered buffer under its current name: what a captured graph has baked in."""
        return tuple((n, t.data_ptr(), tuple(t.shape)) for n, t in self.dh.gpu_arrays.items())

    def _capture_two_steps(self, unit=None):
        """Two steps (two fused PAIRS of steps when ``unit`` is given) as one CUDA graph (a step that swaps buffers is only
        periodic with period 2).  Capturing executes
        the steps' host side — the swaps — but no kernel, so the registry is put back afterwards; a step sequence that is
        not back at the same buffer roles after two steps (a three-buffer rotation) cannot be replayed: None."""
        unit = unit or self._one_step
        torch, dh = self.dh.torch, self.dh
        before = OrderedDict(dh.gpu_arrays)
        roles, n_swaps, n_calls = self._roles(), dh._swap_count, len(dh.call_queue)
        import gc
        stream = torch.cuda.Stream(dh.device)
        stream.wait_stream(torch.cuda.current_stream(dh.device))
        g, periodic = None, False
        # no cyclic garbage collection while the stream is capturing: a collected object that owns CUDA resources (an older
        # graph, an event) would be destroyed in the middle of the capture and invalidate it (torch.cuda.graph collects
        # once BEFORE it begins capturing for the same reason)
        gc_was_on = gc.isenabled()
        gc.disable()
        try:
            with torch.cuda.stream(stream):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream):
                    unit()
                    unit()
            periodic = self._roles() == roles
            self.capture_error = None
        except Exception as exc:         # a failed capture is not fatal: the loop issues its steps eagerly
            chain = [exc] + ([exc.__context__] if exc.__context__ is not None else [])
            self.capture_error = ' <- '.join('%s: %s' % (type(e).__name__, str(e).splitlines()[0] if str(e) else '') for e in chain)
            g = None
        finally:
            if gc_was_on:
                gc.enable()
            torch.cuda.current_stream(dh.device).wait_stream(stream)
            dh.gpu_arrays.clear()
            dh.gpu_arrays.update(before)
            dh._swap_count = n_swaps
            del dh.call_queue[n_calls:]
        return g if periodic else None

    def run(self, time_steps=1):
        """Like graph_datahandling.py:181-190: the calls of the steps are not appended to the data handling's queue one by
        one; the queue gets ONE ``('TimeloopRun', time_steps, steps)`` entry."""
        torch, dh = self.dh.torch, self.dh
        former_queue = dh.call_queue
        dh.call_queue = []
        swaps_per_step = None
        try:
            for f in self._pre:
                f()
            graph_ok = (self.use_cuda_graph and dh.dec.world_size == 1 and torch.cuda.is_available()
                        and all(t.is_cuda for t in dh.gpu_arrays.values()))
            done = 0
            fused = self.fused_pair() if time_steps >= 2 else None
            if fused is not None:
                # two time steps per launch (f-1); `per` = time steps one unit advances
                unit, per = (lambda: self._one_pair(fused)), 2
            else:
                unit, per = self._one_step, 1
            self.fused_last_run = fused is not None
            if graph_ok and time_steps >= 4 * per:
                # warm up (NVRTC / module load must not happen during capture)
                n0 = dh._swap_count
                unit()
                unit()
                swaps_per_step = (dh._swap_count - n0) // 2
                done = 2 * per
                # a graph bakes the buffer pointers in: it is only valid for the roles it was captured with (an odd
                # number of steps in an earlier run, an external swap or a replaced array all change them)
                roles = (self._roles(), per)
                if roles not in self._graphs:
                    if len(self._graphs) >= self.max_cached_graphs:
                        self._graphs.clear()
                    self._graphs[roles] = self._capture_two_steps(unit)
                graph = self._graphs[roles]
                while graph is not None and done + 2 * per <= time_steps:
                    graph.replay()
                    done += 2 * per
            while done + per <= time_steps:
                unit()
                done += per
            for _ in range(time_steps - done):        # the odd last step of a fused run
                self._one_step()
            self.time_steps_run += time_steps
            for f in self._post:
                f()
        finally:
            recorded = self._step_record if self._step_record is not None else tuple(self._single_step_asts)
            dh.call_queue = former_queue
            dh._record(('TimeloopRun', time_steps, recorded))
        return swaps_per_step


class SlabStencilOp:
    """Forward + adjoint of one ``AutoDiffOp`` on this rank's slab — what ``bench.py`` times.

    ``local_shape`` is the owned (ghost-free) shape per rank; the global field is ``world_size`` such slabs stacked
    along dim 0."""

    def __init__(self, op, local_shape, rank=0, world_size=1, device=None, backend='nccl', tuning=None, scalars=None,
                 peer_halo=False):
        import torch
        self.torch = torch
        self.op = op
        self.rank, self.world = rank, world_size
        scalars = dict(scalars or {})
        self.device = device
        self.fwd = CompiledKernel(op.forward_ast_gpu, tuning)
        self.bwd = CompiledKernel(op.backward_ast_gpu, tuning)
        g = 0
        if world_size > 1:
            for ir in (op.forward_ast_gpu, op.backward_ast_gpu):
                g = max(g, max(ir.max_halo[0]))
        global_shape = (local_shape[0] * world_size,) + tuple(local_shape[1:])
        self.dh = SlabDataHandling(global_shape, rank, world_size, g, device, backend, peer_halo=peer_halo)
        self.exchange_kind = ('ncclSend/ncclRecv via psad_halo_exchange on a comm stream, overlapped with interior planes'
                              if backend == 'nccl' else 'torch.distributed P2P')
        if self.dh.peer is not None:
            self.exchange_kind = ('peer halos: ghost planes staged by the stencil kernel\'s own TMA loads from the neighbouring '
                                  'GPUs\' arrays (CUDA IPC, NVLink), one launch per kernel, per-rank launch counters')
        self.local_shape = tuple(local_shape)
        names = OrderedDict()
        for f in list(op.forward_fields) + list(op.backward_fields):
            names.setdefault(f.name, f)
        for n, f in names.items():
            self.dh.add_array(n, dtype=f.dtype.numpy_dtype)
        self.fwd_halo = _exchanged_inputs(op.forward_ast_gpu, self.dh.dec)
        self.bwd_halo = _exchanged_inputs(op.backward_ast_gpu, self.dh.dec)
        _check_scalars((self.fwd, self.bwd), scalars)
        self.scalars = scalars
        self.fwd_scalars = {s_: scalars[s_] for s_ in self.fwd.scalars}
        self.bwd_scalars = {s_: scalars[s_] for s_ in self.bwd.scalars}
        self._fn = None

    def randomize(self, generator):
        """Synthetic inputs: forward inputs ~ U(0.1, 1), upstream gradients ~ N(0, 1)."""
        for f in self.op.forward_input_fields:
            self.dh.owned(f.name).copy_(self.torch.rand(self.local_shape, generator=generator, device=self.device,
                                                        dtype=self.dh.gpu_arrays[f.name].dtype) * 0.9 + 0.1)
        for f in self.op.backward_input_fields:
            if f not in self.op.forward_input_fields:
                self.dh.owned(f.name).copy_(self.torch.randn(self.local_shape, generator=generator, device=self.device,
                                                             dtype=self.dh.gpu_arrays[f.name].dtype))
        if self.dh.peer is not None:
            self.dh.peer.dirty = True         # written outside the launch sequence: fence before the next launch

    def forward(self):
        self.dh.run_kernel(self.fwd, halo_fields=self.fwd_halo, **self.fwd_scalars)

    def backward(self):
        self.dh.run_kernel(self.bwd, halo_fields=self.bwd_halo, **self.bwd_scalars)

    def variants(self):
        return {'forward': self.fwd.last_variant, 'adjoint': self.bwd.last_variant}

    # -- end-to-end with host buffers ----------------------------------------------------------------------------
    def end_to_end(self, steps, barrier, copy_baseline=True):
        """Same metric through the public operator for HOST buffers (``HostStreamedOp``): every step uploads the forward
        inputs and the upstream gradients of this rank's slab from pinned host memory in chunks of planes, runs forward +
        adjoint per chunk and downloads the outputs and the input gradients — upload, kernels and download of consecutive
        chunks overlap on three streams, every rank streams its own slab (one pinned buffer per field), and the planes
        next to a neighbouring rank are exchanged GPU to GPU.  ``copy_baseline``: also time the bare copies of the same
        bytes (H2D on one stream, D2H on another) — the ceiling the host memory / PCIe fabric sets for this step."""
        torch = self.torch
        if self._fn is None:
            self._fn = HostStreamedOp(self.op, self.local_shape, self.device, rank=self.rank, world_size=self.world,
                                      exchanger=self.dh.exchanger if self.world > 1 else None,
                                      kernels=(self.fwd, self.bwd))
            self._host = {n: torch.empty(self.local_shape, dtype=self.dh.gpu_arrays[n].dtype, pin_memory=True)
                          for n in self._fn.fields}
            for n in self._fn.input_names:
                self._host[n].copy_(self.dh.owned(n))
        streamed = self._fn
        h_in = {n: self._host[n] for n in streamed.input_names}
        h_out = {n: self._host[n] for n in streamed.output_names}

        def step():
            streamed(h_in, h_out, **self.scalars)

        def timed(fn, n):
            fn()
            barrier()
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            for _ in range(n):
                fn()
            end.record()
            barrier()
            return start.elapsed_time(end) / n

        result = dict(ms_per_step=timed(step, steps), h2d=streamed.h2d_bytes, d2h=streamed.d2h_bytes,
                      chunks=streamed.n_chunks, chunk_planes=streamed.chunk)
        # the streamed results against the resident kernels on the same inputs (outside the timed region): a few planes of
        # every output — first and last plane of the slab (next to the neighbouring ranks when N > 1) and the planes
        # around two chunk boundaries — bit for bit
        self.forward()
        self.backward()
        torch.cuda.synchronize() if torch.cuda.is_available() else None
        st = streamed.starts
        n0 = self.local_shape[0]
        planes = sorted({0, n0 - 1} | {p for b_ in (st[1:2] + st[-1:]) for p in (b_ - 1, b_) if 0 <= p < n0})
        result['checked_planes'] = planes
        result['matches_resident'] = all(bool(torch.equal(self._host[n][p].to(self.device), self.dh.owned(n)[p]))
                                         for n in streamed.output_names for p in planes)
        if copy_baseline:
            if getattr(self, '_copy_streams', None) is None:
                self._copy_streams = (torch.cuda.Stream(self.device), torch.cuda.Stream(self.device))
            s_up, s_dn = self._copy_streams
            dev_in = [self.dh.owned(n) for n in streamed.input_names]
            dev_out = [self.dh.owned(n) for n in streamed.output_names]

            def copies():
                cur = torch.cuda.current_stream(self.device)
                s_up.wait_stream(cur)
                s_dn.wait_stream(cur)
                with torch.cuda.stream(s_up):
                    for n, d in zip(streamed.input_names, dev_in):
                        d.copy_(self._host[n], non_blocking=True)
                with torch.cuda.stream(s_dn):
                    for n, d in zip(streamed.output_names, dev_out):
                        self._host[n].copy_(d, non_blocking=True)
                cur.wait_stream(s_up)
                cur.wait_stream(s_dn)
            saved = [d.clone() for d in dev_in]       # the uploads overwrite the resident inputs: put them back afterwards
            try:
                result['copy_only_ms'] = timed(copies, max(1, steps))
            finally:
                for d, s_ in zip(dev_in, saved):
                    d.copy_(s_)
        return result


class HostStreamedOp:
    """Forward + adjoint of an ``AutoDiffOp`` on fields that live in (pinned) HOST memory, streamed through the GPU.

    The reference's Function copies whole tensors with ``.cuda()`` inside ``forward`` (backends/_torch_native.py:47-49),
    which serialises H2D, compute and D2H.  Here the fields are cut into chunks of planes along dim 0 (the same slab
    decomposition as the multi-GPU path, with the chunks of one GPU playing the role of the ranks): chunk k+1 is
    uploaded on a copy-in stream while chunk k is computed and chunk k-1 is downloaded on a copy-out stream, so the
    PCIe link runs in both directions at once and the kernels hide behind it.  A chunk's ghost planes are its neighbours'
    planes of the (contiguous) host array; the ``2g`` planes two consecutive chunks share are copied from the previous
    chunk's device buffer, so every input plane crosses PCIe exactly once.  Global boundary handling is the same range
    logic as ``SlabDecomposition``.
    """

    def __init__(self, op, shape, device=None, chunk_planes=None, stages=3, tuning=None, ramp=True, rank=0, world_size=1,
                 exchanger=None, kernels=None):
        """``rank`` / ``world_size`` / ``exchanger`` (a ``HaloExchanger`` of a decomposition with the same ranks): ``shape``
        is then THIS RANK'S slab of a field split along dim 0, each rank streams its own slab from its own host memory,
        and the ``g`` planes next to a neighbouring rank are uploaded first and exchanged GPU to GPU (one small grouped
        send / receive per input field per call), so a chunk at a slab border finds its ghost planes on the device."""
        import torch
        self.torch = torch
        self.op = op
        self.shape = tuple(int(s) for s in shape)
        self.rank, self.world = int(rank), int(world_size)
        self.exchanger = exchanger
        if self.world > 1 and exchanger is None:
            raise ValueError('HostStreamedOp on %d ranks needs a HaloExchanger' % self.world)
        self.global_shape = (self.shape[0] * self.world,) + self.shape[1:]
        self.device = torch.device(device if device is not None else ('cuda', torch.cuda.current_device()))
        self.fwd, self.bwd = kernels if kernels is not None else (CompiledKernel(op.forward_ast_gpu, tuning),
                                                                    CompiledKernel(op.backward_ast_gpu, tuning))
        self.g = max(max(ir.max_halo[0]) for ir in (op.forward_ast_gpu, op.backward_ast_gpu))
        plane_bytes = int(np.prod(self.shape[1:])) * max(f.dtype.itemsize for f in op.forward_fields)
        if chunk_planes is None:
            chunk_planes = max(4 * max(1, self.g), min(self.shape[0], (192 << 20) // max(1, plane_bytes)))
        self.chunk = int(min(chunk_planes, self.shape[0]))
        # Chunk sizes: full chunks in the middle, a quarter and a half chunk at either end — the pipeline fills with the
        # upload of the FIRST chunk and drains with the download of the LAST one, so those are kept short (the planes
        # shared by consecutive chunks are copied on the device, extra chunks cost two launches each).
        self.sizes = self._chunk_sizes(self.shape[0], self.chunk, max(1, 2 * self.g)) if ramp else \
            [min(self.chunk, self.shape[0] - z) for z in range(0, self.shape[0], self.chunk)]
        self.starts = [sum(self.sizes[:i]) for i in range(len(self.sizes))]
        self.n_chunks = len(self.sizes)
        self.stages = int(stages)
        fields = OrderedDict()
        for f in list(op.forward_fields) + list(op.backward_fields):
            fields.setdefault(f.name, f)
        self.fields = fields
        written = {f.name for f in op.forward_output_fields} | {f.name for f in op.backward_output_fields}
        self.input_names = [n for n in fields if n not in written]
        self.output_names = [n for n in fields if n in written]
        buf_shape = (self.chunk + 2 * self.g,) + self.shape[1:]
        self.buffers = [{n: torch.empty(buf_shape, dtype=numpy_dtype_to_torch(f.dtype.numpy_dtype), device=self.device)
                         for n, f in fields.items()} for _ in range(self.stages)]
        # [planes received from below | first g planes | last g planes | planes received from above] per input field
        self.edges = ({n: torch.zeros((4 * self.g,) + self.shape[1:], dtype=self.buffers[0][n].dtype, device=self.device)
                       for n in self.input_names} if (self.world > 1 and self.g > 0) else None)
        self.s_in, self.s_cmp, self.s_out = (torch.cuda.Stream(self.device) for _ in range(3))
        self.ev_in = [torch.cuda.Event() for _ in range(self.stages)]
        self.ev_cmp = [torch.cuda.Event() for _ in range(self.stages)]
        self.ev_out = [torch.cuda.Event() for _ in range(self.stages)]
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self._range_cache = {}

    @staticmethod
    def _chunk_sizes(n0, chunk, smallest):
        """Sizes summing to ``n0``: ``chunk // 4, chunk // 2, chunk, ..., chunk, chunk // 2, chunk // 4`` (ends no smaller than
        ``smallest`` planes; fields too short for the ramp are cut uniformly)."""
        q, h = max(smallest, chunk // 4), max(smallest, chunk // 2)
        if n0 < 2 * (q + h) + chunk or q >= h or h >= chunk:
            return [min(chunk, n0 - z) for z in range(0, n0, chunk)]
        middle = n0 - 2 * (q + h)
        n_mid = -(-middle // chunk)
        base, rem = divmod(middle, n_mid)
        return [q, h] + [base + (1 if i < rem else 0) for i in range(n_mid)] + [h, q]

    def _ranges(self, kernel, z0, n_k):
        key = (id(kernel), z0, n_k)      # one dict per (kernel, chunk), reused every call: the launch path keys on it
        if key not in self._range_cache:
            self._range_cache[key] = self._make_range(kernel, z0, n_k)
        return self._range_cache[key]

    def _make_range(self, kernel, z0, n_k):
        ir = kernel.ir   # the chunk's ghost planes are filled from the host array, so one launch covers it
        return slab_ranges(self.global_shape, self.rank * self.shape[0] + z0, n_k, self.g, False, False, ir.boundary,
                           ir.ghost_layers, ir.ndim)[0]

    def __call__(self, host_in, host_out, **scalars):
        """``host_in``: name -> pinned CPU tensor for every input field (forward inputs and ``diff<out>`` gradients);
        ``host_out``: name -> pinned CPU tensor receiving every output (forward outputs and ``diff<in>``);
        ``scalars``: values of the free scalar symbols of the kernels."""
        torch = self.torch
        _check_scalars((self.fwd, self.bwd), scalars)
        g, C, N0 = self.g, self.chunk, self.shape[0]
        cur = torch.cuda.current_stream(self.device)
        start = torch.cuda.Event()
        start.record(cur)
        for s_ in (self.s_in, self.s_cmp, self.s_out):
            s_.wait_event(start)
        self.h2d_bytes = self.d2h_bytes = 0
        has_lo, has_hi = self.rank > 0, self.rank < self.world - 1
        if self.edges is not None:
            # the planes the neighbouring ranks need go up first and are exchanged GPU to GPU on the upload stream; they
            # cross PCIe a second time with their chunk (2 g planes per field: 0.4 % of a 1024-plane slab)
            with torch.cuda.stream(self.s_in):
                for n in self.input_names:
                    e = self.edges[n]
                    e[g:2 * g].copy_(host_in[n][:g], non_blocking=True)
                    e[2 * g:3 * g].copy_(host_in[n][N0 - g:N0], non_blocking=True)
                    self.h2d_bytes += 2 * g * host_in[n][0].numel() * host_in[n].element_size()
                    if self.exchanger.backend == 'nccl':
                        self.exchanger.exchange_planes(e[g:2 * g], e[:g], e[2 * g:3 * g], e[3 * g:], self.s_in.cuda_stream)
                    else:
                        self.exchanger.exchange_planes(e[g:2 * g], e[:g], e[2 * g:3 * g], e[3 * g:])
        for k in range(self.n_chunks):
            st = k % self.stages
            buf = self.buffers[st]
            z0, n_k = self.starts[k], self.sizes[k]
            lo, hi = max(0, z0 - g), min(N0, z0 + n_k + g)
            with torch.cuda.stream(self.s_in):
                if k >= self.stages:
                    self.s_in.wait_event(self.ev_out[st])      # the buffer's previous chunk has been downloaded
                    self.s_in.wait_event(self.ev_cmp[st])
                # planes [z0 - g, z0 + g) are already on the device — the previous chunk uploaded them into ITS buffer (same
                # stream, so ordered; a different ring slot, so intact): a device copy instead of a second trip over PCIe
                prev = self.buffers[(k - 1) % self.stages] if (k > 0 and g > 0 and self.stages > 1) else None
                for n in self.input_names:
                    dst = buf[n]
                    off = lo - (z0 - g)
                    if off > 0:
                        if has_lo:
                            dst[:off].copy_(self.edges[n][g - off:g], non_blocking=True)     # the lower rank's last planes
                        else:
                            dst[:off].zero_()                   # planes below the domain: the 'zeros' boundary
                    up_lo = lo
                    if prev is not None:
                        n_prev = self.sizes[k - 1]
                        dst[:2 * g].copy_(prev[n][n_prev:n_prev + 2 * g], non_blocking=True)
                        up_lo = min(N0, z0 + g)                 # the previous chunk's buffer reached plane z0 + g
                    if hi > up_lo:
                        dst[up_lo - (z0 - g):off + (hi - lo)].copy_(host_in[n][up_lo:hi], non_blocking=True)
                        self.h2d_bytes += (hi - up_lo) * host_in[n][0].numel() * host_in[n].element_size()
                    if off + (hi - lo) < n_k + 2 * g:
                        if has_hi:
                            m = n_k + 2 * g - (off + (hi - lo))
                            dst[off + (hi - lo):n_k + 2 * g].copy_(self.edges[n][3 * g:3 * g + m], non_blocking=True)
                        else:
                            dst[off + (hi - lo):n_k + 2 * g].zero_()
                self.ev_in[st].record(self.s_in)
            with torch.cuda.stream(self.s_cmp):
                self.s_cmp.wait_event(self.ev_in[st])
                if k >= self.stages:
                    self.s_cmp.wait_event(self.ev_out[st])
                for kern in (self.fwd, self.bwd):
                    for f in kern.ir.output_fields:
                        if f in kern.ir.input_fields:       # ``+=`` form: accumulates onto a zero-initialised output
                            buf[f.name].zero_()
                    views = {f.name: buf[f.name][:n_k + 2 * g] for f in kern.fields}
                    kern(**views, **{s_: scalars[s_] for s_ in kern.scalars}, _range=self._ranges(kern, z0, n_k))
                self.ev_cmp[st].record(self.s_cmp)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_cmp[st])
                for n in self.output_names:
                    host_out[n][z0:z0 + n_k].copy_(buf[n][g:g + n_k], non_blocking=True)
                    self.d2h_bytes += n_k * host_out[n][0].numel() * host_out[n].element_size()
                self.ev_out[st].record(self.s_out)
        done = torch.cuda.Event()
        done.record(self.s_out)
        cur.wait_event(done)
        cur.wait_event(self.ev_cmp[(self.n_chunks - 1) % self.stages])
