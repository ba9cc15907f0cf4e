"""GPU: bfloat16 fields (bf16 storage, fp32 arithmetic) through the autograd Function, run_steps, TimeLoop with CUDA-graph
replay, a periodic slab, the generic kernel and ``data_type='double'``, against the fp64 oracle evaluated on the bf16
inputs (tolerances as tests/test_bf16_replay.py: 4e-3 of the largest value per launch, 8e-3 for time loops against the
oracle rounded to bf16 after every step).  The range test is why bf16 exists next to fp16: values around 1e6 and
gradients around 1e-9 survive bf16 storage, while fp16 overflows the one and flushes the other to zero.  Every test
checks that native launches happened."""
import numpy as np
import pytest

from oracle import evaluate
from pystencils_autodiff_b200 import runtime
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
from pystencils_autodiff_b200.configs import make_config

pytestmark = pytest.mark.gpu

BF16_TOL = 4e-3
STEPS_TOL = 8e-3
FUSE_REASON = 'bfloat16 fields: fused pairs not implemented'


@pytest.fixture(autouse=True)
def _bf16_words_in_cpu_dry_run(monkeypatch, tmp_path_factory):
    """The CPU dry run of these bodies (tests/dryrun_plugin.py) replays launches on numpy arrays, which cannot hold
    bfloat16: there the kernels get int16 views of the same storage, and the replays compile against the shim copies with
    the bfloat16 host stand-ins of tests/test_bf16_replay.py.  Does nothing on a GPU."""
    import torch
    call = CompiledKernel.__call__
    if call.__qualname__ == 'ReplayKernel.__call__':
        from test_bf16_replay import use_bf16_shims
        use_bf16_shims(tmp_path_factory.getbasetemp() / 'bf16_shims_dry_run', monkeypatch)

        def words(self, **kw):
            return call(self, **{k: (v.detach().view(torch.int16) if isinstance(v, torch.Tensor) and v.dtype == torch.bfloat16
                                     else v) for k, v in kw.items()})
        monkeypatch.setattr(CompiledKernel, '__call__', words)
    yield


def _launches():
    """Native kernel launches so far (in the CPU dry run of these bodies, tests/dryrun_plugin.py: replayed launches)."""
    return runtime.launch_count() + len(getattr(CompiledKernel, 'launches', ()))


def _bf(a):
    """float array -> bf16 CUDA tensor (each value rounded to bf16)."""
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(torch.bfloat16).cuda()


def _np(t):
    """bf16 tensor -> float64 numpy (exact)."""
    return t.detach().float().cpu().numpy().astype(np.float64)


def _rel_err(got, ref):
    return float(np.abs(np.asarray(got, dtype=np.float64) - ref).max() / max(1e-300, np.abs(ref).max()))


def _rounded_steps(assigns, u, steps, bh, src='u', dst='out'):
    import torch
    ref = u.astype(np.float64)
    for _ in range(steps):
        ref = torch.from_numpy(evaluate(assigns, {src: ref}, bh)[dst]).to(torch.bfloat16).double().numpy()
    return ref


def _function_run(name, shape, bh, in_scale=1.0, grad_scale=1.0, seed=1):
    """Forward and backward of the Function on bf16 tensors; returns (op, outputs, input tensors, fp64 oracle values)."""
    import torch
    op = make_config(name, shape=shape, dtype='bfloat16', boundary_handling=bh)
    op64 = make_config(name, shape=shape, dtype='float64', boundary_handling=bh)
    fn = op.create_tensorflow_op(backend='torch_native', use_cuda=True)
    rng = np.random.default_rng(seed)
    tens = [_bf(rng.uniform(0.5, 1.5, size=shape) * in_scale).requires_grad_(True) for f in op.forward_input_fields]
    gts = [_bf(rng.uniform(-1, 1, size=shape) * grad_scale) for f in op.forward_output_fields]
    n0 = _launches()
    outs = fn.apply(*tens)
    torch.autograd.backward(outs, gts)
    torch.cuda.synchronize()
    assert _launches() - n0 == 2
    assert fn.forward_kernel.last_variant == 'march' and fn.backward_kernel.last_variant == 'march'
    ins = {f.name: _np(t) for f, t in zip(op.forward_input_fields, tens)}
    fwd = evaluate(op64.forward_assignments, ins, bh)
    bwd_in = dict(ins)
    bwd_in.update({'diff' + f.name: _np(g) for f, g in zip(op.forward_output_fields, gts)})
    bwd = evaluate(op64.backward_assignments, bwd_in, bh)
    for f, o in zip(op.forward_output_fields, outs):
        assert o.dtype == torch.bfloat16
        assert _rel_err(_np(o), fwd[f.name]) <= BF16_TOL, (f.name,)
    for f, t in zip(op.forward_input_fields, tens):
        assert t.grad.dtype == torch.bfloat16
        assert _rel_err(_np(t.grad), bwd['diff' + f.name]) <= BF16_TOL, ('diff' + f.name,)
    return op, outs, tens, gts


@pytest.mark.parametrize('name, shape', [('c2', (72, 264)), ('c3', (13, 37, 136)), ('c4', (9, 21, 136)),
                                         ('c5', (3, 27, 136))])
@pytest.mark.parametrize('bh', ['zeros', None])
def test_bf16_function_forward_and_backward(name, shape, bh):
    """The torch_native Function on bfloat16 tensors: bf16 outputs and bf16 gradients from the march kernels."""
    _function_run(name, shape, bh)


def test_bf16_range_beyond_float16():
    """C3 with inputs around 1e6 and an upstream gradient around 1e-9 (a mean() over a large field): bf16 outputs and
    gradients are non-zero and within 4e-3 of the oracle.  The same gradient stored as float16 is all zeros."""
    import torch
    op, outs, tens, gts = _function_run('c3', (13, 37, 136), 'zeros', in_scale=1e6, grad_scale=1e-9, seed=5)
    assert outs[0].float().abs().min().item() > 1e5
    assert tens[0].grad.float().abs().max().item() > 1e-10
    assert (gts[0].float().abs() > 0).float().mean().item() > 0.99
    assert torch.count_nonzero(gts[0].half()).item() == 0          # fp16 flushes every one of these gradients to zero
    assert torch.isinf(outs[0].half()).all()                        # and overflows every one of these values


def test_bf16_float32_op_refuses_bf16_tensors():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('the dtype check belongs to the native launch path, which the CPU dry run replaces')
    k32 = CompiledKernel(make_config('c2', shape=(8, 128)).forward_ast_gpu)
    x = torch.zeros((8, 128), dtype=torch.bfloat16, device='cuda')
    n0 = _launches()
    with pytest.raises(TypeError, match='expects dtype float32'):
        k32(u=x, out=torch.empty_like(x))
    k32(u=x.float(), out=torch.empty_like(x.float()))
    torch.cuda.synchronize()
    assert _launches() - n0 == 1


def test_bf16_c3_full_size_sampled_blocks():
    """C3 in bf16 at its full size 1024^3: forward and adjoint, checked on sampled blocks (corner, centre, far corner)
    against the oracle evaluated on the block plus its one-cell halo."""
    import torch
    N = 1024
    op = make_config('c3', shape=(N, N, N), dtype='bfloat16')
    fwd, bwd = CompiledKernel(op.forward_ast_gpu), CompiledKernel(op.backward_ast_gpu)
    g = torch.Generator(device='cuda').manual_seed(3)
    u = torch.rand((N, N, N), device='cuda', generator=g).to(torch.bfloat16)
    out = torch.empty_like(u)
    n0 = _launches()
    fwd(u=u, out=out)
    diffu = torch.empty_like(u)
    bwd(diffout=out, diffu=diffu)
    torch.cuda.synchronize()
    assert _launches() - n0 == 2 and fwd.last_variant == 'march' and bwd.last_variant == 'march'
    B = (10, 18, 128)
    for z0, y0, x0 in ((0, 0, 0), (500, 401, 448), (N - B[0], N - B[1], N - B[2])):
        lo = [max(0, c - 1) for c in (z0, y0, x0)]
        hi = [min(N, c + b + 1) for c, b in zip((z0, y0, x0), B)]
        sl = tuple(slice(a, b) for a, b in zip(lo, hi))
        inner = tuple(slice(c - a, c - a + b) for c, a, b in zip((z0, y0, x0), lo, B))
        blk = tuple(slice(c, c + b) for c, b in zip((z0, y0, x0), B))
        ops = make_config('c3', shape=tuple(b - a for a, b in zip(lo, hi)), dtype='float64')
        ref = evaluate(ops.forward_assignments, {'u': _np(u[sl])}, 'zeros')['out'][inner]
        assert _rel_err(_np(out[blk]), ref) <= BF16_TOL, (z0, y0, x0)
        refd = evaluate(ops.backward_assignments, {'diffout': _np(out[sl])}, 'zeros')['diffu'][inner]
        assert _rel_err(_np(diffu[blk]), refd) <= BF16_TOL, (z0, y0, x0)


def test_bf16_data_type_double():
    """``data_type='double'`` on bfloat16 fields: fp64 arithmetic, one rounding from fp64 per stored cell."""
    import torch
    import pystencils_autodiff_b200 as ps
    shape = (9, 30, 136)
    u, out = ps.fields('u, out: bfloat16[%d,%d,%d]' % shape)
    lap = u[1, 0, 0] + u[-1, 0, 0] + u[0, 1, 0] + u[0, -1, 0] + u[0, 0, 1] + u[0, 0, -1] - 6 * u[0, 0, 0]
    op = ps.AutoDiffOp([ps.Assignment(out.center, u.center + 0.1 * lap)], op_name='heat_d', boundary_handling='zeros',
                       data_type='double')
    assert op.forward_ast_gpu.compute_dtype == np.float64
    k = CompiledKernel(op.forward_ast_gpu)
    x = _bf(np.random.default_rng(4).uniform(-1, 1, shape) * 1e-20)
    o = torch.full(shape, float('nan'), dtype=torch.bfloat16, device='cuda')
    n0 = _launches()
    k(u=x, out=o)
    torch.cuda.synchronize()
    assert _launches() - n0 == 1 and k.last_variant == 'march' and 'typedef double CT;' in k.code
    op64 = make_config('c3', shape=shape, dtype='float64')
    ref = evaluate(op64.forward_assignments, {'u': _np(x)}, 'zeros')['out']
    assert _rel_err(_np(o), ref) <= BF16_TOL


def test_bf16_generic_agrees_with_march():
    import torch
    shape = (11, 40, 264)
    op = make_config('c4', shape=shape, dtype='bfloat16')
    k = CompiledKernel(op.forward_ast_gpu)
    x = _bf(np.random.default_rng(6).uniform(-1, 1, shape))
    a, b = torch.empty_like(x), torch.empty_like(x)
    n0 = _launches()
    k(u=x, out=a)
    assert k.last_instance == 'march_nomask'
    k(u=x, out=b, _variant='generic')
    assert k.last_variant == 'generic'
    torch.cuda.synchronize()
    assert _launches() - n0 == 2
    # different summation orders (plane sums vs one FMA chain): at most one bf16 rounding step apart
    assert (a.float() - b.float()).abs().max().item() <= 2.0 ** -7 * a.float().abs().max().item()
    assert (a != b).float().mean().item() < 0.2
    # a strided view takes the generic kernel and gives the same values as the generic kernel on the dense copy
    big = torch.zeros(shape[:2] + (shape[2] + 3,), dtype=torch.bfloat16, device='cuda')
    view = big[:, :, 1:1 + shape[2]]
    view.copy_(x)
    c = torch.empty_like(x)
    k(u=view, out=c)
    assert k.last_variant == 'generic'
    torch.cuda.synchronize()
    assert torch.equal(b, c)


def test_bf16_run_steps_and_timeloop_graph_replay():
    """Single steps only (fused pairs are declined for bf16): T launches for T steps, eager and CUDA-graph replayed TimeLoop
    bit-identical to run_steps, all against the oracle rounded to bf16 after every step."""
    import torch
    from pystencils_autodiff_b200.datahandling import SlabDataHandling
    shape, T = (12, 40, 264), 5
    op = make_config('c3', shape=shape, dtype='bfloat16')
    op64 = make_config('c3', shape=shape, dtype='float64')
    k = CompiledKernel(op.forward_ast_gpu)
    assert k.fused_steps_reason() == FUSE_REASON
    u0 = _bf(np.random.default_rng(9).uniform(-1, 1, shape))
    u0_64 = _np(u0)
    n0 = _launches()
    out = k.run_steps(u0.clone(), T)
    torch.cuda.synchronize()
    assert _launches() - n0 == T
    with pytest.raises(ValueError, match='bfloat16'):
        k.run_steps(u0.clone(), T, fuse=True)
    ref = _rounded_steps(op64.forward_assignments, u0_64, T, 'zeros')
    assert _rel_err(_np(out), ref) <= STEPS_TOL
    finals = []
    for use_graph in (True, False):
        dh = SlabDataHandling(shape, 0, 1, 0, device='cuda:0')
        dh.add_arrays('u, out', dtype='bfloat16')
        dh.owned('u').copy_(u0)
        tl = dh.create_timeloop(use_cuda_graph=use_graph)
        tl.add_call(k, {})
        tl.swap('u', 'out')
        n0 = _launches()
        tl.run(T)
        tl.run(T)
        torch.cuda.synchronize()
        assert not tl.fused_last_run and tl.time_steps_run == 2 * T
        if use_graph and torch.cuda.is_available():          # (the CPU dry run of this body has no CUDA graphs)
            assert tl._graphs and all(g is not None for g in tl._graphs.values())
        if not use_graph:
            assert _launches() - n0 == 2 * T      # (graph replays are not counted as launches)
        finals.append(dh.owned('u').clone())
        dh2 = SlabDataHandling(shape, 0, 1, 0, device='cuda:0')
        dh2.add_arrays('u, out', dtype='bfloat16')
        tl2 = dh2.create_timeloop(fuse_steps=True)
        tl2.add_call(k, {})
        tl2.swap('u', 'out')
        with pytest.raises(ValueError, match='bfloat16'):
            tl2.fused_pair()
    assert torch.equal(finals[0], finals[1])
    ref = _rounded_steps(op64.forward_assignments, u0_64, 2 * T, 'zeros')
    assert _rel_err(_np(finals[0]), ref) <= STEPS_TOL
    assert torch.equal(finals[0], k.run_steps(u0.clone(), 2 * T))


def test_bf16_periodic_single_rank():
    """One rank, periodic along dim 0 (the rank is its own neighbour): bf16 ghost planes wrapped around by the exchange."""
    import torch
    from pystencils_autodiff_b200.datahandling import SlabDataHandling
    gshape, T = (16, 24, 136), 3
    dh = SlabDataHandling(gshape, 0, 1, 1, device='cuda:0', periodic=True)
    dh.add_arrays('u, out', dtype='bfloat16')
    op_l = make_config('c3', shape=dh.dec.local_shape, dtype='bfloat16')
    k = CompiledKernel(op_l.forward_ast_gpu)
    u0 = _bf(np.random.default_rng(11).uniform(-1, 1, gshape))
    dh.owned('u').copy_(u0)
    n0 = _launches()
    dh.run_steps(k, T)
    torch.cuda.synchronize()
    n = _launches() - n0
    assert n >= T and n % T == 0
    got = dh.gather_array('u')
    assert got.dtype == np.float32
    op_w = make_config('c3', shape=(gshape[0] + 2,) + gshape[1:], dtype='float64')
    ref = _np(u0)
    for _ in range(T):
        wrapped = np.concatenate([ref[-1:], ref, ref[:1]], axis=0)
        out = evaluate(op_w.forward_assignments, {'u': wrapped}, 'zeros')['out'][1:-1]
        ref = torch.from_numpy(out).to(torch.bfloat16).double().numpy()
    assert _rel_err(got, ref) <= STEPS_TOL
