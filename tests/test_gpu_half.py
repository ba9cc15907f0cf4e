"""GPU: float16 fields (fp16 storage, fp32 arithmetic) through the autograd Function, run_steps, TimeLoop with CUDA-graph
replay, a periodic slab, the generic kernel and ``data_type='double'``, against the fp64 oracle evaluated on the fp16
inputs (tolerances as tests/test_half_replay.py: 5e-4 of the largest value per step, 1e-3 for time loops against the
oracle rounded to fp16 after every step).  Every test checks that native launches happened."""
import numpy as np
import pytest

from oracle import evaluate
from pystencils_autodiff_b200 import runtime
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
from pystencils_autodiff_b200.configs import make_config

pytestmark = pytest.mark.gpu

F16 = np.float16
HALF_TOL = 5e-4
STEPS_TOL = 1e-3


def _launches():
    """Native kernel launches so far (in the CPU dry run of these bodies, tests/dryrun_plugin.py: replayed launches)."""
    return runtime.launch_count() + len(getattr(CompiledKernel, 'launches', ()))


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _rel_err(got, ref):
    return float(np.abs(np.asarray(got, dtype=np.float64) - ref).max() / max(1e-30, np.abs(ref).max()))


def _rounded_steps(assigns, u, steps, bh, src='u', dst='out'):
    ref = u.astype(np.float64)
    for _ in range(steps):
        ref = evaluate(assigns, {src: ref}, bh)[dst].astype(F16).astype(np.float64)
    return ref


@pytest.mark.parametrize('name, shape', [('c2', (72, 264)), ('c3', (13, 37, 136)), ('c4', (9, 21, 136)),
                                         ('c5', (3, 27, 136))])
@pytest.mark.parametrize('bh', ['zeros', None])
def test_half_function_forward_and_backward(name, shape, bh):
    """The torch_native Function on float16 tensors: fp16 outputs and fp16 gradients from the march kernels."""
    import torch
    op = make_config(name, shape=shape, dtype='float16', boundary_handling=bh)
    op64 = make_config(name, shape=shape, dtype='float64', boundary_handling=bh)
    fn = op.create_tensorflow_op(backend='torch_native', use_cuda=True)
    rng = np.random.default_rng(1)
    ins = {f.name: rng.uniform(0.5, 1.5, size=shape).astype(F16) for f in op.forward_input_fields}
    grads = {f.name: rng.uniform(-1, 1, size=shape).astype(F16) for f in op.forward_output_fields}
    tens = [_t(ins[f.name]).requires_grad_(True) for f in op.forward_input_fields]
    n0 = _launches()
    outs = fn.apply(*tens)
    torch.autograd.backward(outs, [_t(grads[f.name]) for f in op.forward_output_fields])
    torch.cuda.synchronize()
    assert _launches() - n0 == 2
    assert fn.forward_kernel.last_variant == 'march' and fn.backward_kernel.last_variant == 'march'
    fwd = evaluate(op64.forward_assignments, {k: v.astype(np.float64) for k, v in ins.items()}, bh)
    for f, o in zip(op.forward_output_fields, outs):
        assert o.dtype == torch.float16
        assert _rel_err(o.detach().cpu().numpy(), fwd[f.name]) <= HALF_TOL, (f.name,)
    bwd_in = {k: v.astype(np.float64) for k, v in ins.items()}
    bwd_in.update({'diff' + k: v.astype(np.float64) for k, v in grads.items()})
    bwd = evaluate(op64.backward_assignments, bwd_in, bh)
    for f, t in zip(op.forward_input_fields, tens):
        assert t.grad.dtype == torch.float16
        assert _rel_err(t.grad.cpu().numpy(), bwd['diff' + f.name]) <= HALF_TOL, ('diff' + f.name,)


def test_half_c3_full_size_sampled_blocks():
    """C3 in fp16 at its full size 1024^3: forward and adjoint, checked on sampled blocks (corner, centre, far corner)
    against the oracle evaluated on the block plus its one-cell halo."""
    import torch
    N = 1024
    op = make_config('c3', shape=(N, N, N), dtype='float16')
    fwd, bwd = CompiledKernel(op.forward_ast_gpu), CompiledKernel(op.backward_ast_gpu)
    g = torch.Generator(device='cuda').manual_seed(3)
    u = torch.rand((N, N, N), device='cuda', generator=g).half()
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
        blk_u = u[sl].float().cpu().numpy().astype(np.float64)
        # the block's own border is the array border only where the block touches it: evaluate on the haloed block
        ops = make_config('c3', shape=blk_u.shape, dtype='float64')
        ref = evaluate(ops.forward_assignments, {'u': blk_u}, 'zeros')['out'][inner]
        got = out[tuple(slice(c, c + b) for c, b in zip((z0, y0, x0), B))].float().cpu().numpy()
        assert _rel_err(got, ref) <= HALF_TOL, (z0, y0, x0)
        blk_o = out[sl].float().cpu().numpy().astype(np.float64)
        refd = evaluate(ops.backward_assignments, {'diffout': blk_o}, 'zeros')['diffu'][inner]
        gotd = diffu[tuple(slice(c, c + b) for c, b in zip((z0, y0, x0), B))].float().cpu().numpy()
        assert _rel_err(gotd, refd) <= HALF_TOL, (z0, y0, x0)


def test_half_data_type_double():
    """``data_type='double'`` on float16 fields: fp64 arithmetic, one rounding from fp64 per stored cell."""
    import torch
    import pystencils_autodiff_b200 as ps
    shape = (9, 30, 136)
    u, out = ps.fields('u, out: float16[%d,%d,%d]' % shape)
    lap = u[1, 0, 0] + u[-1, 0, 0] + u[0, 1, 0] + u[0, -1, 0] + u[0, 0, 1] + u[0, 0, -1] - 6 * u[0, 0, 0]
    op = ps.AutoDiffOp([ps.Assignment(out.center, u.center + 0.1 * lap)], op_name='heat_d', boundary_handling='zeros',
                       data_type='double')
    assert op.forward_ast_gpu.compute_dtype == np.float64
    k = CompiledKernel(op.forward_ast_gpu)
    x = np.random.default_rng(4).uniform(-1, 1, shape).astype(F16)
    o = torch.full(shape, float('nan'), dtype=torch.float16, device='cuda')
    n0 = _launches()
    k(u=_t(x), out=o)
    torch.cuda.synchronize()
    assert _launches() - n0 == 1 and k.last_variant == 'march' and 'typedef double CT;' in k.code
    op64 = make_config('c3', shape=shape, dtype='float64')
    ref = evaluate(op64.forward_assignments, {'u': x.astype(np.float64)}, 'zeros')['out']
    assert _rel_err(o.cpu().numpy(), ref) <= HALF_TOL


def test_half_generic_agrees_with_march():
    import torch
    shape = (11, 40, 264)
    op = make_config('c4', shape=shape, dtype='float16')
    k = CompiledKernel(op.forward_ast_gpu)
    x = _t(np.random.default_rng(6).uniform(-1, 1, shape).astype(F16))
    a, b = torch.empty_like(x), torch.empty_like(x)
    n0 = _launches()
    k(u=x, out=a)
    assert k.last_instance == 'march_nomask'
    k(u=x, out=b, _variant='generic')
    assert k.last_variant == 'generic'
    torch.cuda.synchronize()
    assert _launches() - n0 == 2
    # different summation orders (plane sums vs one FMA chain): at most one fp16 rounding step apart
    assert (a.float() - b.float()).abs().max().item() <= 2.0 ** -10 * a.float().abs().max().item()
    assert (a != b).float().mean().item() < 0.05
    # a strided view takes the generic kernel and gives the same halves as the generic kernel on the dense copy
    big = torch.zeros(shape[:2] + (shape[2] + 3,), dtype=torch.float16, device='cuda')
    view = big[:, :, 1:1 + shape[2]]
    view.copy_(x)
    c = torch.empty_like(x)
    k(u=view, out=c)
    assert k.last_variant == 'generic'
    torch.cuda.synchronize()
    assert torch.equal(b, c)


def test_half_run_steps_and_timeloop_graph_replay():
    """Single steps only (fused pairs are declined for fp16): T launches for T steps, eager and CUDA-graph replayed TimeLoop
    bit-identical to run_steps, all against the oracle rounded to fp16 after every step."""
    import torch
    from pystencils_autodiff_b200.datahandling import SlabDataHandling
    shape, T = (12, 40, 264), 5
    op = make_config('c3', shape=shape, dtype='float16')
    op64 = make_config('c3', shape=shape, dtype='float64')
    k = CompiledKernel(op.forward_ast_gpu)
    assert k.fused_steps_reason() == 'float16 fields: fused pairs not implemented'
    u0 = np.random.default_rng(9).uniform(-1, 1, shape).astype(F16)
    n0 = _launches()
    out = k.run_steps(_t(u0), T)
    torch.cuda.synchronize()
    assert _launches() - n0 == T
    with pytest.raises(ValueError, match='float16'):
        k.run_steps(_t(u0), T, fuse=True)
    ref = _rounded_steps(op64.forward_assignments, u0, T, 'zeros')
    assert _rel_err(out.cpu().numpy(), ref) <= STEPS_TOL
    finals = []
    for use_graph in (True, False):
        dh = SlabDataHandling(shape, 0, 1, 0, device='cuda:0')
        dh.add_arrays('u, out', dtype=F16)
        dh.owned('u').copy_(_t(u0))
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
        dh2.add_arrays('u, out', dtype=F16)
        tl2 = dh2.create_timeloop(fuse_steps=True)
        tl2.add_call(k, {})
        tl2.swap('u', 'out')
        with pytest.raises(ValueError, match='float16'):
            tl2.fused_pair()
    assert torch.equal(finals[0], finals[1])
    ref = _rounded_steps(op64.forward_assignments, u0, 2 * T, 'zeros')
    assert _rel_err(finals[0].cpu().numpy(), ref) <= STEPS_TOL
    assert torch.equal(finals[0], k.run_steps(_t(u0), 2 * T))


def test_half_periodic_single_rank():
    """One rank, periodic along dim 0 (the rank is its own neighbour): fp16 ghost planes wrapped around by the exchange."""
    import torch
    from pystencils_autodiff_b200.datahandling import SlabDataHandling
    gshape, T = (16, 24, 136), 3
    dh = SlabDataHandling(gshape, 0, 1, 1, device='cuda:0', periodic=True)
    dh.add_arrays('u, out', dtype=F16)
    op_l = make_config('c3', shape=dh.dec.local_shape, dtype='float16')
    k = CompiledKernel(op_l.forward_ast_gpu)
    u0 = np.random.default_rng(11).uniform(-1, 1, gshape).astype(F16)
    dh.owned('u').copy_(_t(u0))
    n0 = _launches()
    dh.run_steps(k, T)
    torch.cuda.synchronize()
    n = _launches() - n0
    assert n >= T and n % T == 0
    got = dh.owned('u').cpu().numpy()
    op_w = make_config('c3', shape=(gshape[0] + 2,) + gshape[1:], dtype='float64')
    ref = u0.astype(np.float64)
    for _ in range(T):
        wrapped = np.concatenate([ref[-1:], ref, ref[:1]], axis=0)
        ref = evaluate(op_w.forward_assignments, {'u': wrapped}, 'zeros')['out'][1:-1].astype(F16).astype(np.float64)
    assert _rel_err(got, ref) <= STEPS_TOL
