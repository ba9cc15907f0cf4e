#!/usr/bin/env python
"""bench.py — forward+adjoint stencil throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2|c4|c5] [--dump-outputs DIR]

One "step" = one forward kernel + one adjoint kernel over the whole field (per GPU: weak scaling, every rank owns
a slab of the workload's full single-GPU shape; ghost planes are exchanged with the neighbours before each kernel
when N > 1).  Prints ONE JSON line on rank 0.  The headline workload is C3 (the configuration BASELINE.json shards over
1/2/4/8 GPUs); at N = 1 the same line carries the other named configurations (``workloads``: C2, C4, C5, each with its own
timed region, roofline and clocks), the ``torch.autograd.Function`` path (``function_path``), full-size parity against the
CPU oracle (``parity``) and the end-to-end legs with host buffers (``e2e``, ``e2e_plugin``).  See DESIGN.md "Measurement".

The benchmark writes nothing into the source tree, which may be read-only: kernels it has to compile at run time (NVRTC
cubins, the oracle's C kernels) go to a temporary directory that is removed at exit; the cubins build() compiled into the
tree are used from there.
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

METRIC = 'forward+adjoint Mcell-updates/s'
UNIT = 'Mcell-updates/s'
WORKLOADS = {
    'c2': 'C2: 2-D 5-point diffusion step + adjoint, 8192x8192 fp32, zeros boundary',
    'c3': 'C3: 3-D 7-point heat-equation stencil + adjoint, 1024^3 fp32 per GPU (slab-sharded along dim 0), zeros boundary',
    'c4': 'C4: 3-D 27-point stencil + adjoint, 768^3 fp64, zeros boundary',
    'c5': 'C5: 2-D TV-denoising gradient + adjoint, batch 16 of 4096x4096 fp32, zeros boundary',
}
DTYPE = {'c2': 'f32', 'c3': 'f32', 'c4': 'f64', 'c5': 'f32'}
TOL = {'f32': 1e-6, 'f64': 1e-12}          # north_star: <= 1e-6 relative in fp32, <= 1e-12 in fp64
# The one stated exception (INTEGRATION.md section 5, profiles/r2_c5_accuracy.md): the ADJOINT of the TV-denoising gradient
# evaluated in fp32 arithmetic.  Its coefficients grow like 1/|grad u|^3; over the 268 M cells of C5 a few dozen cells with
# vanishing gradients (conditioning ~10, terms of +-1e3 cancelling) end up 1e-6 .. 4e-6 away from the double-precision
# reference in the max norm whatever the evaluation order or the accuracy of the reciprocal root (measured: a Newton-refined
# root changes nothing), while 99.99999 % of the cells are within 5e-7.  pystencils' default arithmetic for fp32 fields is
# double: AutoDiffOp(..., data_type='double') reproduces it and is checked at 1e-6 beside this (``double_arithmetic``).
TOL_OVERRIDE = {('c5', 'adjoint'): 1e-5}
BAD_CLOCK_REASONS = {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}
DUMP_BYTES = 60 * 10**6          # --dump-outputs: payload of all arrays together, under 64 MB with the .npy headers


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c3', choices=sorted(WORKLOADS))
    ap.add_argument('--shape', type=int, nargs='*', default=None, help='override the per-GPU field shape')
    ap.add_argument('--e2e-steps', type=int, default=3)
    ap.add_argument('--strong', action='store_true',
                    help='strong scaling: the workload shape is the GLOBAL field, split along dim 0 over the ranks '
                         '(default: weak scaling, every rank owns the full workload shape)')
    ap.add_argument('--halo', default='auto', choices=['auto', 'nccl', 'peer'],
                    help='N > 1: ghost planes by NCCL exchange, read by the kernels from the neighbours\' memory (peer), or '
                         'whichever was measured to win for this slab size (auto)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true', help='skip the end-to-end leg (diagnostic runs)')
    ap.add_argument('--only-headline', action='store_true', help='skip the extra N = 1 legs (workloads, function path, parity)')
    ap.add_argument('--cpu-shape', type=int, nargs='*', default=None, help='CPU arm: sample shape (default: the full workload)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed (the forward outputs and the input '
                         'gradients of the headline workload) as DIR/<field>.npy; arrays over %d MB in all are replaced '
                         'by a fixed seeded sample of their elements' % (DUMP_BYTES // 10**6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes what the GPU path computed: it needs --impl ours')
    return args


def use_private_build_dirs():
    """Kernels compiled at run time go to a temporary directory, removed at exit (see the module docstring).  The cubins
    build() left in the package's cache are linked into the temporary cache, so they are not compiled again."""
    tmp = tempfile.mkdtemp(prefix='psad_bench_')
    atexit.register(shutil.rmtree, tmp, True)
    if 'PSAD_CACHE_DIR' not in os.environ:
        cubins = os.path.join(tmp, 'cubin')
        os.makedirs(cubins)
        built = os.path.join(ROOT, 'pystencils_autodiff_b200', '_cubin_cache')
        for name in (os.listdir(built) if os.path.isdir(built) else []):
            if name.endswith('.cubin'):
                os.symlink(os.path.join(built, name), os.path.join(cubins, name))
        os.environ['PSAD_CACHE_DIR'] = cubins
    os.environ.setdefault('PSAD_ORACLE_BUILD_DIR', os.path.join(tmp, 'oracle'))


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, power and clock-event (throttle) reasons sampled DURING the timed region (B200_PROFILING.md recipe).

    NVML — the library behind nvidia-smi — polled from a thread without sleeping (a C2 timed region is 4 ms long: the
    ``nvidia-smi -lms`` subprocess of round 1 delivered no sample at all inside it); falls back to that subprocess when the
    NVML binding is missing.  Samples are stamped on arrival and ``stop(t0, t1)`` keeps the ones inside the region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.index = index
        self.samples = []          # (t, sm_mhz, power_w, reasons)
        self.max_mhz = None
        self.proc = None
        self.thread = None
        self.running = False
        self.source = None

    def start(self):
        self.running = True
        try:
            if os.environ.get('PSAD_BENCH_NO_NVML'):
                raise ImportError('NVML polling disabled')
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(visible.split(',')[self.index]) if visible and visible.split(',')[self.index].strip().isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = [('hw_slowdown', pynvml.nvmlClocksEventReasonHwSlowdown),
                    ('hw_thermal_slowdown', pynvml.nvmlClocksEventReasonHwThermalSlowdown),
                    ('sw_thermal_slowdown', pynvml.nvmlClocksEventReasonSwThermalSlowdown),
                    ('sw_power_cap', pynvml.nvmlClocksEventReasonSwPowerCap)]

            def poll():
                while self.running:
                    try:
                        mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        watts = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                    except Exception:
                        break
                    self.samples.append((time.perf_counter(), mhz, watts, [n for n, b in bits if mask & b]))
            self.source = 'nvml'
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.source = 'nvidia-smi -lms 20'
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

        def pump():
            for line in self.proc.stdout:
                parts = [p.strip() for p in line.split(',')]
                if len(parts) < 7:
                    continue
                try:
                    self.max_mhz = float(parts[1])
                    self.samples.append((time.perf_counter(), float(parts[0]), float(parts[2]),
                                         [n for n, v in zip(names, parts[3:7]) if v.lower().startswith('active')]))
                except ValueError:
                    continue
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self, t0=None, t1=None):
        self.running = False
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)
        if self.source is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no NVML binding and no nvidia-smi'], 'samples': 0}
        inside = [s_ for s_ in self.samples if (t0 is None or s_[0] >= t0) and (t1 is None or s_[0] <= t1)]
        note = None
        if not inside and self.samples:            # region shorter than the sampling period: the samples nearest to it
            mid = 0.5 * ((t0 or 0) + (t1 or 0))
            inside = sorted(self.samples, key=lambda s_: abs(s_[0] - mid))[:3]
            note = 'no sample inside the region: nearest samples used'
        sm = sorted(s_[1] for s_ in inside)
        reasons = sorted({r for s_ in inside for r in s_[3]})
        out = {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.max_mhz, 'sm_min_mhz': sm[0] if sm else None,
               'power_w_max': max((s_[2] for s_ in inside), default=None), 'reasons': reasons, 'samples': len(inside),
               'source': self.source}
        if note:
            out['note'] = note
        return out


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs: burst copy bandwidth, best of 10)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def bind_to_gpu_numa_node(device_index):
    """N > 1: keep this rank's threads — and with them the pinned host buffers it allocates (first touch) — on the NUMA node
    its GPU hangs off, so eight ranks do not pull their host traffic through one socket.  Returns what was done."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(device_index)
        bus = '%04x:%02x:%02x.0' % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open('/sys/bus/pci/devices/%s/numa_node' % bus) as fh:
            node = int(fh.read().strip())
        if node < 0:
            return {'numa_node': None, 'note': 'the platform reports no NUMA node for %s' % bus}
        with open('/sys/devices/system/node/node%d/cpulist' % node) as fh:
            cpus = set()
            for part in fh.read().strip().split(','):
                lo, _, hi = part.partition('-')
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {'numa_node': node, 'cpus': len(allowed), 'pci': bus}
    except Exception as exc:
        return {'numa_node': None, 'note': '%s: %s' % (type(exc).__name__, exc)}


# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_run(workload, steps, warmup, shape=None):
    """The reference's CPU implementation of the path, restated (oracle/cgen.py, 'fast' flavour = pystencils'
    cpujit flag set, OpenMP over all host threads), timed on the workload's full shape unless a sample shape is given."""
    import numpy as np
    import torch
    from oracle.cgen import compile_c
    from pystencils_autodiff_b200.configs import CONFIG_SHAPES, make_config

    full = tuple(CONFIG_SHAPES[workload]['shape'])
    shape = tuple(shape or full)
    threads = host_threads()
    os.environ['OMP_NUM_THREADS'] = str(threads)
    op = make_config(workload, shape=shape, boundary_handling='zeros')
    fwd = compile_c(op.forward_assignments, 'zeros', op.op_name + '_forward_cpu', 'fast')
    bwd = compile_c(op.backward_assignments, 'zeros', op.op_name + '_backward_cpu', 'fast')
    arrays = {}
    gen = torch.Generator().manual_seed(0)
    for f in sorted(set(op.forward_fields) | set(op.backward_fields), key=str):
        # torch.rand: multi-threaded fill (numpy's generator takes ~8 s per GiB-element array on one core)
        dt = getattr(torch, np.dtype(f.dtype.numpy_dtype).name)
        arrays[f.name] = (torch.rand(shape, generator=gen, dtype=dt) * 0.9 + 0.1).numpy()
    cells = int(np.prod(shape))

    def step():
        fwd(**{n: arrays[n] for n in fwd.field_names})
        bwd(**{n: arrays[n] for n in bwd.field_names})

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(1, steps)
    what = 'the full workload shape' if shape == full else 'a %s sample of the workload' % 'x'.join(map(str, shape))
    return dict(value=cells / dt / 1e6, unit=UNIT, cores=threads, kind='port', shape=list(shape), full_shape=shape == full,
                sample='%s: forward+adjoint over %s (%s = %d cells), %d timed passes after %d warm-up, gcc -Ofast -march=native '
                       '-fopenmp, restated pystencils CPU path (pystencils itself is not installable here)'
                       % (workload, what, 'x'.join(map(str, shape)), cells, steps, warmup)), dt


def main_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    base, dt = cpu_reference_run(args.workload, args.steps, max(1, args.warmup), args.cpu_shape or args.shape)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': base['value'], 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': DTYPE[args.workload], 'data': 'synthetic',
        'config': {'workload': WORKLOADS[args.workload], 'per_gpu_shape': base['shape'], 'cpu_sample': base['sample']},
        'cpu_baseline': base,
        'e2e': {'value': base['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------------
class Env:
    """Process-wide state of the GPU arm."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local_rank = int(os.environ.get('LOCAL_RANK', '0'))
        if not torch.cuda.is_available():
            raise RuntimeError('bench.py --impl ours needs a CUDA device: this backend has no CPU fallback')
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device('cuda', self.local_rank)
        self.numa = bind_to_gpu_numa_node(self.local_rank) if self.world > 1 else None
        if self.world > 1:
            os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
            dist.init_process_group('nccl', device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        if self.world == 1:
            return [float(v) for v in values]
        t = self.torch.tensor(list(values), device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]


def measure_resident(env, wl, shape, steps, warmup, cooldown_s=0.0, halo='auto'):
    """The device-timed metric for one workload: K steps of forward + adjoint launches through the C ABI on resident
    arrays, CUDA events, barrier on both sides, max over ranks.  Returns ``(result dict, slab, op)``."""
    import numpy as np
    from pystencils_autodiff_b200 import runtime
    from pystencils_autodiff_b200.configs import make_config
    from pystencils_autodiff_b200.datahandling import SlabStencilOp
    torch = env.torch
    t_setup0 = time.perf_counter()
    op = make_config(wl, shape=shape, boundary_handling='zeros')
    slab = SlabStencilOp(op, local_shape=shape, rank=env.rank, world_size=env.world, device=env.dev,
                         peer_halo={'auto': 'auto', 'nccl': False, 'peer': True}[halo])
    setup_ms = {'symbolic_and_emit_ms': (time.perf_counter() - t_setup0) * 1e3}
    cells = int(np.prod(shape))
    b_fwd = op.forward_ast_gpu.bytes_per_cell()
    b_bwd = op.backward_ast_gpu.bytes_per_cell()
    g = torch.Generator(device=env.dev)
    g.manual_seed(1234 + env.rank)
    slab.randomize(g)

    def step(events=None):
        if events is not None:
            events[0].record()
        slab.forward()
        if events is not None:
            events[1].record()
        slab.backward()
        if events is not None:
            events[2].record()

    # the first step pays for NVRTC (or a cubin-cache hit), module load and — N > 1 — the NCCL connections: reported
    # separately (SURVEY section 8d), never inside a timed region
    t_first0 = time.perf_counter()
    step()
    env.barrier()
    setup_ms['first_step_ms'] = (time.perf_counter() - t_first0) * 1e3
    warmup = max(3, warmup)
    # per-kernel durations: CUDA events around the forward and the adjoint launch on every `stride`-th timed step (an
    # event between two 90 us kernels costs a few us of GPU idle time, so not on every step)
    stride = 1 if steps < 8 else (4 if steps < 40 else 8)

    def timed_region():
        if cooldown_s:
            env.barrier()
            time.sleep(cooldown_s)       # start from an idle GPU: this pool's B200s power-cap within ~150 ms of streaming
        for _ in range(warmup):
            step()
        n0 = runtime.launch_count()
        clocks = ClockSampler(env.local_rank)
        if env.rank == 0:
            clocks.start()
        evs = {i: [torch.cuda.Event(enable_timing=True) for _ in range(3)] for i in range(0, steps, stride)}
        env.barrier()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        t_host0 = time.perf_counter()
        for i in range(steps):
            step(evs.get(i))
        host_ms_ = (time.perf_counter() - t_host0) * 1e3 / steps   # CPU time spent issuing one step
        end.record()
        env.barrier()
        t_host1 = time.perf_counter()
        clk_ = clocks.stop(t_host0, t_host1) if env.rank == 0 else None
        return (start.elapsed_time(end), sum(e[0].elapsed_time(e[1]) for e in evs.values()) / len(evs),
                sum(e[1].elapsed_time(e[2]) for e in evs.values()) / len(evs), host_ms_, clk_,
                runtime.launch_count() - n0, len(evs))

    ms_total, t_fwd, t_bwd, host_ms, clk, launches, n_samples = timed_region()
    # a run that saw a hardware / thermal slowdown is rejected and measured again, once (sw_power_cap is kept and noted)
    retry = torch.tensor([1 if (env.rank == 0 and clk and BAD_CLOCK_REASONS & set(clk.get('reasons', []))) else 0], device=env.dev)
    if env.world > 1:
        env.dist.all_reduce(retry, op=env.dist.ReduceOp.MAX)
    if int(retry.item()):
        first_reasons = clk.get('reasons') if clk else None
        time.sleep(2.0)
        ms_total, t_fwd, t_bwd, host_ms, clk, launches, n_samples = timed_region()
        if clk is not None:
            clk['remeasured_after'] = first_reasons
    ms_total, t_fwd, t_bwd = env.max_over_ranks([ms_total, t_fwd, t_bwd])
    ms_step = ms_total / steps
    peak, peak_src = measured_peaks()
    achieved = cells * b_fwd / (t_fwd * 1e-3) / 1e9
    pair = cells * (b_fwd + b_bwd) / ((t_fwd + t_bwd) * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tpath):
        with open(tpath) as fh:
            traffic = json.load(fh).get(wl, {}).get('forward_dram_bytes_per_launch')
    res = {
        'value': cells * env.world / (ms_step * 1e-3) / 1e6, 'unit': UNIT, 'ms_per_step': ms_step, 'steps': steps, 'warmup': warmup,
        'dtype': DTYPE[wl],
        'config': {'workload': WORKLOADS[wl], 'per_gpu_shape': list(shape), 'cells_per_gpu': cells,
                   'bytes_per_cell': {'forward': b_fwd, 'adjoint': b_bwd},
                   'l2': 'inputs larger than L2 (%.2f GB per field vs 126 MB): no flush needed'
                         % (cells * op.forward_input_fields[0].dtype.itemsize / 1e9),
                   'kernel_variants': slab.variants(),
                   'halo_exchange': slab.exchange_kind if env.world > 1 else 'none (1 GPU)'},
        'roofline': {'bound': 'hbm', 'kernel': op.forward_ast_gpu.function_name, 'achieved': achieved, 'peak': peak,
                     'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                     'forward_ms': t_fwd, 'adjoint_ms': t_bwd, 'kernel_timing_samples': n_samples,
                     'pair_achieved': pair, 'pair_frac': pair / peak, 'pair_frac_of_8000_nominal': pair / 8000.0},
        'clocks': clk, 'gpu_launches': launches, 'setup': setup_ms, 'host_issue_ms_per_step': host_ms,
    }
    return res, slab, op


def dump_outputs(env, op, slab, out_dir):
    """``--dump-outputs``: the arrays the timed step hands its caller — the forward outputs and the adjoint's input
    gradients of this rank's slab — as ``out_dir/<field>.npy`` in their own dtype (``<field>.rank<r>.npy`` when N > 1).
    Every rank gets DUMP_BYTES / N: when its arrays exceed that together, each is replaced by its elements at the same
    seeded, sorted flat indices in every run (``numpy.random.default_rng(0)``), so that two builds of the project can be
    compared output for output."""
    import numpy as np
    torch = env.torch
    names = list(dict.fromkeys(f.name for f in list(op.forward_output_fields) + list(op.backward_output_fields)))
    arrays = {n: slab.dh.owned(n) for n in names}
    budget = DUMP_BYTES // env.world
    sample = sum(t.numel() * t.element_size() for t in arrays.values()) > budget
    suffix = '.rank%d' % env.rank if env.world > 1 else ''
    os.makedirs(out_dir, exist_ok=True)
    torch.cuda.synchronize()
    for name, t in arrays.items():
        if sample:
            k = budget // len(arrays) // t.element_size()
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), size=k))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + suffix + '.npy'), t.cpu().numpy())


def function_path(env, op, slab, steps):
    """The path the north-star names: ``Function.apply`` + backward on RESIDENT tensors — output and gradient allocation
    (``torch.empty``), ``save_for_backward``, the autograd engine and the ctypes call all inside the timed region —
    timed with CUDA events and with the wall clock."""
    import numpy as np
    torch = env.torch
    fn = op.create_tensorflow_op(backend='torch_native', use_cuda=True)
    xs = [slab.dh.owned(f.name).detach().requires_grad_(True) for f in op.forward_input_fields]
    grads = tuple(slab.dh.owned(f.name) for f in op.backward_input_fields
                  if f not in op.forward_input_fields and f not in op.forward_output_fields)
    cells = int(np.prod(slab.local_shape))

    def step():
        outs = fn.apply(*xs)
        return torch.autograd.grad(outs, xs, grad_outputs=grads, allow_unused=True)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record()
    for _ in range(steps):
        step()
    b.record()
    t_issue = time.perf_counter() - t0
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t0
    ms = a.elapsed_time(b) / steps
    return {'ms_per_step': ms, 'value': cells / (ms * 1e-3) / 1e6, 'unit': UNIT, 'wall_ms_per_step': t_wall * 1e3 / steps,
            'host_issue_ms_per_step': t_issue * 1e3 / steps, 'steps': steps,
            'api': 'Op = AutoDiffOp(...).create_tensorflow_op(backend="torch_native", use_cuda=True); outs = Op.apply(*inputs); '
                   'torch.autograd.grad(outs, inputs, upstream) — resident CUDA tensors, allocation included'}


def oracle_parity(env, wl, op, slab, kernels=None, tol_override=True):
    """Full-size parity against the CPU oracle (``oracle/cgen.py``, 'strict' flavour: the restated pystencils loop nest in
    double precision, no contraction): blocks of planes of the workload-sized outputs the resident kernels just produced —
    first planes, a block in the middle, last planes — recomputed from the same inputs (the block plus its halo planes are
    brought to the host) and compared norm-wise.  The oracle is the checker here, never the thing measured."""
    import numpy as np
    from oracle.cgen import compile_c
    torch = env.torch
    if kernels is None:
        slab.forward()
        slab.backward()
    else:                                   # another arithmetic mode of the same operator on the slab's arrays
        for k in kernels:
            k(**{f.name: slab.dh.gpu_arrays[f.name] for f in k.fields}, **{s_: slab.scalars[s_] for s_ in k.scalars})
    torch.cuda.synchronize()
    n0 = slab.local_shape[0]
    tol = TOL[DTYPE[wl]]
    worst, checked, per_kernel, ok, tols = 0.0, [], {}, True, {}
    for assigns, ir, tag in ((op.forward_assignments, op.forward_ast_gpu, 'forward'),
                             (op.backward_assignments, op.backward_ast_gpu, 'adjoint')):
        g = max(ir.max_halo[0])
        nb = max(1, min(4, n0 // 8)) if ir.ndim == 3 else max(1, min(64, n0 // 8))
        if g == 0:
            nb = 1                                                    # independent slices along dim 0 (C5: one image)
        blocks = sorted({(0, min(n0, nb)), (max(0, n0 // 2 - nb // 2), min(n0, n0 // 2 - nb // 2 + nb)), (max(0, n0 - nb), n0)})
        kern = compile_c(assigns, 'zeros', '%s_%s_parity' % (op.op_name, tag), 'strict')
        out_names = {f.name for f in ir.output_fields}
        err_k = 0.0
        for z0, z1 in blocks:
            lo, hi = max(0, z0 - g), min(n0, z1 + g)
            bufs = {}
            for f in ir.all_fields:
                dev = slab.dh.owned(f.name)
                bufs[f.name] = (np.zeros((hi - lo,) + tuple(dev.shape[1:]), dtype=f.dtype.numpy_dtype) if f.name in out_names
                                else dev[lo:hi].cpu().numpy())
            kern(**{n: bufs[n] for n in kern.field_names})
            for name in out_names:
                ref = bufs[name][z0 - lo:z1 - lo]            # the block's own planes: their halo planes were inside [lo, hi)
                got = slab.dh.owned(name)[z0:z1].cpu().numpy()
                scale = max(float(np.abs(ref).max()), 1e-300)
                err_k = max(err_k, float(np.abs(got.astype(np.float64) - ref.astype(np.float64)).max()) / scale)
            checked.append([tag, z0, z1])
        per_kernel[tag] = err_k
        tols[tag] = TOL_OVERRIDE.get((wl, tag), tol) if tol_override else tol
        ok = ok and err_k <= tols[tag]
        worst = max(worst, err_k)
    return {'oracle': 'oracle/cgen.py strict (C restatement of the pystencils CPU loop nest, double precision)',
            'max_rel_err': worst, 'per_kernel': per_kernel, 'tolerance': tol, 'tolerance_per_kernel': tols, 'ok': bool(ok),
            'blocks_dim0': checked, 'shape': list(slab.local_shape)}


def double_arithmetic(env, wl, slab, shape):
    """The reference's arithmetic for fp32 fields (pystencils ``data_type='double'``: loads promoted, everything computed in
    double, rounded on store) on the same arrays: parity at the unrelaxed 1e-6 and what it costs."""
    from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
    from pystencils_autodiff_b200.configs import make_config
    torch = env.torch
    op = make_config(wl, shape=shape, boundary_handling='zeros', data_type='double')
    ks = (CompiledKernel(op.forward_ast_gpu), CompiledKernel(op.backward_ast_gpu))
    res = oracle_parity(env, wl, op, slab, kernels=ks, tol_override=False)
    out = {'parity': {k: res[k] for k in ('max_rel_err', 'per_kernel', 'tolerance', 'ok')}}
    for k, tag in zip(ks, ('forward_ms', 'adjoint_ms')):
        arrs = {f.name: slab.dh.gpu_arrays[f.name] for f in k.fields}
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k(**arrs)
        a.record()
        for _ in range(5):
            k(**arrs)
        b.record()
        torch.cuda.synchronize()
        out[tag] = a.elapsed_time(b) / 5
    return out


def sharded_parity(env, op, slab):
    """N > 1: the planes around every slab boundary, recomputed UNSHARDED on rank 0 from the gathered input planes and
    compared bit for bit with what the ranks computed from exchanged ghost planes."""
    import numpy as np
    torch, dist = env.torch, env.dist
    slab.forward()
    slab.backward()
    torch.cuda.synchronize()
    n0 = slab.local_shape[0]
    result = {'sharded_equals_unsharded': True, 'boundaries': env.world - 1, 'planes_per_boundary': {}, 'mismatches': []}
    for ir, tag in ((op.forward_ast_gpu, 'forward'), (op.backward_ast_gpu, 'adjoint')):
        g = max(ir.max_halo[0])
        if g == 0:
            result['planes_per_boundary'][tag] = 0       # no reach along dim 0: nothing is exchanged
            continue
        m = g + 1                                         # owned planes checked on each side of a boundary
        w = m + g                                         # input planes needed on each side
        if n0 < w:
            continue
        kern = slab.fwd if tag == 'forward' else slab.bwd
        ins = [f.name for f in ir.input_fields]
        outs = [f.name for f in ir.output_fields]
        # every rank contributes [first w | last w] input planes and [first m | last m] output planes
        packs = {}
        for name, k in [(n, w) for n in ins] + [(n, m) for n in outs]:
            t = slab.dh.owned(name)
            mine = torch.cat([t[:k], t[n0 - k:]]).contiguous()
            parts = [torch.empty_like(mine) for _ in range(env.world)]
            dist.all_gather(parts, mine)
            packs[name] = (parts, k)
        if env.rank == 0:
            for r in range(env.world - 1):
                small = {}
                for name in ins:
                    parts, k = packs[name]
                    small[name] = torch.cat([parts[r][k:], parts[r + 1][:k]]).contiguous()        # 2 w planes across the cut
                for name in outs:
                    small[name] = torch.empty_like(small[ins[0]])
                kern(**small, **{s_: slab.scalars[s_] for s_ in kern.scalars})
                for name in outs:
                    parts, k = packs[name]
                    want = torch.cat([parts[r][k:], parts[r + 1][:k]])
                    got = small[name][g:g + 2 * m]
                    if not torch.equal(got, want):
                        result['sharded_equals_unsharded'] = False
                        result['mismatches'].append([tag, name, r, float((got - want).abs().max())])
            torch.cuda.synchronize()
        result['planes_per_boundary'][tag] = 2 * m
    flag = torch.tensor([1 if result['sharded_equals_unsharded'] else 0], device=env.dev)
    dist.broadcast(flag, src=0)
    result['sharded_equals_unsharded'] = bool(int(flag.item()))
    return result


def plugin_e2e(env, op, slab, steps):
    """The reference-style call with HOST data (backends/_torch_native.py:47-49 copies whole tensors with ``.cuda()``):
    pinned host tensors -> ``.cuda()`` -> ``Op.apply`` -> backward -> results copied back to pinned host tensors; whole-tensor
    copies, nothing overlapped.  Beside ``e2e`` (the chunk-streamed operator) it shows what the streaming buys."""
    import numpy as np
    torch = env.torch
    fn = op.create_tensorflow_op(backend='torch_native', use_cuda=True)
    host = slab._host
    in_names = [f.name for f in op.forward_input_fields]
    out_names = [f.name for f in op.forward_output_fields]
    grad_names = [f.name for f in op.backward_input_fields if f not in op.forward_input_fields and f not in op.forward_output_fields]
    din_names = [f.name for f in op.backward_output_fields]
    cells = int(np.prod(slab.local_shape))

    def step():
        xs = [host[n].cuda(non_blocking=True).requires_grad_(True) for n in in_names]
        outs = fn.apply(*xs)
        ups = tuple(host[n].cuda(non_blocking=True) for n in grad_names)
        gin = torch.autograd.grad(outs, xs, grad_outputs=ups, allow_unused=True)
        for n, t in zip(out_names, outs):
            host[n].copy_(t, non_blocking=True)
        for n, t in zip(din_names, [g_ for g_ in gin if g_ is not None]):
            host[n].copy_(t, non_blocking=True)

    step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    return {'value': cells / (ms * 1e-3) / 1e6, 'unit': UNIT, 'ms_per_step': ms, 'steps': steps, 'timing': 'wall clock',
            'api': 'pinned host tensors -> .cuda() -> Op.apply -> torch.autograd.grad -> .copy_ to pinned host (whole tensors)'}


def extra_legs(env, wl, op, slab, args, with_fused=True):
    """The diagnostics beside a workload's headline number (N = 1): fused forward+adjoint, fused pairs of steps."""
    torch = env.torch
    import numpy as np
    cells = int(np.prod(slab.local_shape))
    out = {}
    # ---- forward and adjoint as ONE launch (AutoDiffOp.fused_kernel_gpu): possible here because the upstream gradient
    # is an input of the step; reported beside the headline, not instead of it
    try:
        fk = op.fused_kernel_gpu
        arrs = {f.name: slab.dh.gpu_arrays[f.name] for f in fk.fields}
        for _ in range(3):
            fk(**arrs)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        f0.record()
        nf = max(5, args.steps // 4)
        for _ in range(nf):
            fk(**arrs)
        f1.record()
        torch.cuda.synchronize()
        fused_ms = f0.elapsed_time(f1) / nf
        out['fused_forward_adjoint'] = {
            'ms_per_step': fused_ms, 'value': cells / (fused_ms * 1e-3) / 1e6, 'unit': UNIT,
            'bytes_per_cell': op.fused_ast_gpu.bytes_per_cell(),
            'note': 'one launch over the union of forward and adjoint assignments (outside the headline timed region)'}
    except NotImplementedError:
        out['fused_forward_adjoint'] = None
    except Exception as exc:
        out['fused_forward_adjoint'] = {'error': '%s: %s' % (type(exc).__name__, exc)}
    # ---- two unrolled steps of the forward stencil as ONE launch (emit_chain.py, SURVEY section 8 f-1) beside two
    # single-step launches; reported next to the headline, not part of it
    steps_info = None
    try:
        fk = slab.fwd
        if fk.fused_steps_reason() is None:
            fin, fout = op.forward_ast_gpu.input_fields[0].name, op.forward_ast_gpu.output_fields[0].name
            g = slab.dh.gpu_arrays
            src, dst, tmp = g[fin], g[fout], g[[n for n in g if n not in (fin, fout)][-1]]
            keep = tmp.clone()

            def _time(fn, n=5):
                for _ in range(3):
                    fn()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a.record()
                for _ in range(n):
                    fn()
                b.record()
                torch.cuda.synchronize()
                return a.elapsed_time(b) / n

            def _two():
                fk(**{fin: src, fout: tmp})
                fk(**{fin: tmp, fout: dst})
            t_two = _time(_two)
            t_x2 = _time(lambda: fk(**{fin: src, fout: dst}, _variant='march_x2'))
            tmp.copy_(keep)
            steps_info = {'two_launches_ms': t_two, 'one_fused_launch_ms': t_x2, 'speedup': t_two / t_x2,
                          'gcell_steps_per_s': 2 * src.numel() / (t_x2 * 1e-3) / 1e9,
                          'used_by_default': True,
                          'note': 'out = S(S(u)) with one read and one write of the field; the default of run_steps() / '
                                  'create_unrolled_torch_op() wherever a pair can be built'}
            # the same through the REFERENCE's time-loop API (GraphDataHandling.TimeLoop: add_call(kernel) + swap(in, out),
            # graph_datahandling.py:152-197): the loop recognises the idiom and issues fused pairs by default
            try:
                keep_src, keep_dst = src.clone(), dst.clone()
                T = 8

                def _loop(fuse):
                    tl = slab.dh.create_timeloop(use_cuda_graph=True, fuse_steps=fuse)
                    tl.add_call(fk, {})
                    tl.swap(fin, fout)
                    tl.run(T)                         # warm-up, graph capture
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    a.record()
                    tl.run(T)
                    tl.run(T)
                    b.record()
                    torch.cuda.synchronize()
                    return a.elapsed_time(b) / (2 * T), tl.fused_last_run, tl.capture_error
                t_single, f_single, err_single = _loop(False)
                t_default, f_default, err_default = _loop(None)
                src.copy_(keep_src)
                dst.copy_(keep_dst)
                del keep_src, keep_dst
                steps_info['time_loop_api'] = {
                    'ms_per_time_step_default': t_default, 'fused_pairs_by_default': bool(f_default),
                    'ms_per_time_step_single_steps': t_single, 'speedup': t_single / t_default, 'time_steps': 2 * T,
                    'cuda_graph_capture_error': err_single or err_default,
                    'api': 'dh.create_timeloop(); tl.add_call(kernel, {}); tl.swap(in, out); tl.run(T)'}
            except Exception as exc:
                steps_info['time_loop_api'] = {'error': '%s: %s' % (type(exc).__name__, exc)}
    except Exception as exc:   # a diagnostic beside the headline must never take the line down
        steps_info = {'error': '%s: %s' % (type(exc).__name__, exc)}
    out['fused_steps'] = steps_info
    return out


def guarded(fn, *a, **kw):
    """A leg beside the headline reports its failure inside its own object instead of killing the line."""
    try:
        return fn(*a, **kw)
    except Exception as exc:
        return {'error': '%s: %s' % (type(exc).__name__, exc)}


def main_ours(args):
    import numpy as np
    from pystencils_autodiff_b200 import runtime
    from pystencils_autodiff_b200.configs import CONFIG_SHAPES
    env = Env()
    torch, dist = env.torch, env.dist
    wl = args.workload
    shape = tuple(args.shape or CONFIG_SHAPES[wl]['shape'])   # per-GPU (local) shape: weak scaling
    if args.strong:
        if shape[0] % env.world:
            raise SystemExit('--strong: dim 0 (%d) must be divisible by the number of GPUs (%d)' % (shape[0], env.world))
        shape = (shape[0] // env.world,) + shape[1:]
    n_launch0 = runtime.launch_count()
    head, slab, op = measure_resident(env, wl, shape, args.steps, args.warmup, halo=args.halo)
    if args.dump_outputs:
        dump_outputs(env, op, slab, args.dump_outputs)     # before the legs below overwrite the arrays
    cells = int(np.prod(shape))

    legs = {}
    if env.world == 1:
        legs.update(extra_legs(env, wl, op, slab, args))
        if not args.only_headline:
            legs['function_path'] = {wl: guarded(function_path, env, op, slab, max(5, args.steps))}
            legs['parity'] = {wl: guarded(oracle_parity, env, wl, op, slab)}
    else:
        legs['parity'] = guarded(sharded_parity, env, op, slab)

    # ---- end to end through the public API with HOST buffers (copies inside the timed region) -------------------
    e2e_error = None
    try:
        if args.no_e2e:
            raise RuntimeError('skipped (--no-e2e)')
        # every rank pins one host buffer per field: refuse (and say so) rather than drive the box out of memory
        need = sum(t.numel() * t.element_size() for t in slab.dh.gpu_arrays.values()) * env.world
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = None
        if avail is not None and need > 0.6 * avail:
            raise MemoryError('the e2e leg pins %.0f GB of host memory over %d ranks, %.0f GB are available'
                              % (need / 1e9, env.world, avail / 1e9))
        e2e = slab.end_to_end(args.e2e_steps, env.barrier)
    except Exception as exc:   # e.g. not enough pinnable host memory: keep the line, say what happened
        e2e_error = '%s: %s' % (type(exc).__name__, exc)
        e2e = {'ms_per_step': float('inf'), 'h2d': 0, 'd2h': 0}
    worst = env.max_over_ranks([e2e['ms_per_step'], e2e.get('copy_only_ms') or 0.0,
                                0.0 if e2e.get('matches_resident', True) else 1.0])
    e2e['ms_per_step'], copy_only_ms, mismatch = worst
    if e2e_error is None and mismatch:
        e2e_error = 'streamed results differ from the resident kernels on planes %s (some rank)' % e2e.get('checked_planes')
    e2e_value = cells * env.world / (e2e['ms_per_step'] * 1e-3) / 1e6 if e2e_error is None else None
    if env.world == 1 and e2e_error is None and not args.only_headline:
        legs['e2e_plugin'] = guarded(plugin_e2e, env, op, slab, 2)

    peer_errors = slab.dh.peer.errors() if slab.dh.peer is not None else None
    slab.dh.close()            # collective: peer-halo mappings of the neighbours' arrays are released before anyone frees them
    if env.rank != 0:
        if env.world > 1:
            dist.destroy_process_group()
        return 0

    line = {
        'metric': METRIC, 'value': head['value'], 'unit': UNIT, 'n_gpus': env.world, 'steps': args.steps, 'warmup': head['warmup'],
        'ms_per_step': head['ms_per_step'], 'higher_is_better': True, 'scaling': 'strong' if args.strong else 'weak',
        'vs_baseline': None, 'dtype': DTYPE[wl], 'data': 'synthetic',
        'config': head['config'],
        'roofline': head['roofline'],
        'clocks': head['clocks'],
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': e2e['h2d'], 'd2h_bytes_per_step': e2e['d2h'],
                'ms_per_step': e2e['ms_per_step'] if e2e_error is None else None, 'steps': args.e2e_steps, 'error': e2e_error,
                'matches_resident': e2e.get('matches_resident'), 'checked_planes': e2e.get('checked_planes'),
                'chunks': e2e.get('chunks'), 'chunk_planes': e2e.get('chunk_planes'),
                'copy_only_ms_per_step': copy_only_ms or None,
                'copy_only_note': 'the same bytes as bare H2D + D2H copies on two streams, max over ranks: what host memory '
                                  'and PCIe allow for this step without any kernel',
                'numa': env.numa,
                'api': 'HostStreamedOp(AutoDiffOp)(host_in, host_out) on every rank: the rank\'s slab of pinned host fields is '
                       'streamed through its GPU in plane chunks, H2D / forward+adjoint kernels / D2H overlapped on three '
                       'streams' + ('; planes next to a neighbouring rank are exchanged GPU to GPU (ncclSend/ncclRecv)'
                                    if env.world > 1 else '')},
        'gpu_launches': head['gpu_launches'],
        'setup': head['setup'],
        'host_issue_ms_per_step': head['host_issue_ms_per_step'],
    }
    if env.world > 1:
        line['halo'] = {'requested': args.halo, 'used': 'peer' if peer_errors is not None else 'nccl', 'peer_wait_timeouts': peer_errors}
    line.update(legs)

    # ---- the other named configurations (BASELINE.json configs 2, 4, 5): own timed region, roofline and clocks each ----
    if env.world == 1 and not args.only_headline and not args.shape and not args.strong:
        del slab
        torch.cuda.empty_cache()
        others = {}
        for w in [w for w in ('c4', 'c2', 'c5') if w != wl]:
            try:
                torch.cuda.empty_cache()
                r, s_w, op_w = measure_resident(env, w, tuple(CONFIG_SHAPES[w]['shape']), args.steps, args.warmup, cooldown_s=1.0)
                r.update(extra_legs(env, w, op_w, s_w, args))
                if w in ('c2', 'c5'):
                    line['function_path'][w] = guarded(function_path, env, op_w, s_w, max(5, args.steps))
                line['parity'][w] = guarded(oracle_parity, env, w, op_w, s_w)
                if w == 'c5':
                    r['double_arithmetic'] = guarded(double_arithmetic, env, w, s_w, tuple(CONFIG_SHAPES[w]['shape']))
                del s_w, op_w
                others[w] = r
            except Exception as exc:
                others[w] = {'error': '%s: %s' % (type(exc).__name__, exc)}
        line['workloads'] = others
        par = line.get('parity', {})
        line['parity_ok'] = bool(par) and all(isinstance(v, dict) and v.get('ok') for v in par.values())
    line['gpu_launches_total'] = runtime.launch_count() - n_launch0
    line['launch_cache'] = dict(zip(('hits', 'misses'), runtime.launch_cache_stats()))

    if not args.no_cpu_baseline and env.world == 1:
        try:
            base, _ = cpu_reference_run(wl, steps=20, warmup=2, shape=args.cpu_shape)
        except Exception as exc:
            base = {'value': None, 'unit': UNIT, 'cores': host_threads(), 'kind': 'port', 'sample': 'failed',
                    'error': '%s: %s' % (type(exc).__name__, exc)}
        line['cpu_baseline'] = base
    print(json.dumps(line), flush=True)
    if env.world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    a = parse_args()
    use_private_build_dirs()
    sys.exit(main_reference(a) if a.impl == 'reference' else main_ours(a))
