"""GPU: the random stencils of tests/stencil_fuzz.py in float16 and bfloat16 (x-halos of 1-4 cells, asymmetric halos,
several input fields with different pads, several outputs, non-linear terms, both boundary modes, ghost layers that are
not a multiple of 4, a ragged last x tile), forward and adjoint, checked cell by cell against the fp64 oracle evaluated on
the exact 16-bit inputs (``stencil_fuzz.check_cells``: half a spacing of the stored type plus the fp32 allowance).

Every kernel runs as the instance a plain launch selects, as the generic kernel, and, where the rows are 16-byte aligned,
as the masked march instance under a launch range whose x bounds cut inside a lane.  Further cases: gradients scaled into
the edge ranges of each type, ``data_type='double'`` (one rounding from fp64, κ = 1e-12), and kernels that mix float16,
bfloat16 and float32 fields.  The CPU replay of the same cases is tests/test_lowp_fuzz_replay.py."""
import numpy as np
import pytest

from oracle import evaluate
from pystencils_autodiff_b200 import runtime
from pystencils_autodiff_b200.backends._torch_native import CompiledKernel
from stencil_fuzz import (DOUBLE_SHAPES, KAPPA, KAPPA_DOUBLE, SCALED, check_outputs, fuzz_case, fuzz_inputs, ragged_range,
                          reached)

pytestmark = pytest.mark.gpu


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


def _launch(k, stored, **kw):
    """One launch of ``k`` on CUDA copies of the stored arrays (bfloat16: uint16 words); returns the arrays after it."""
    import torch

    def dev(a):
        a = a.copy()                 # (the CPU dry run's .cuda() returns the same storage)
        return torch.from_numpy(a.view(np.int16)).view(torch.bfloat16).cuda() if a.dtype == np.uint16 else \
            torch.from_numpy(a).cuda()

    def host(t):
        t = t.cpu()
        return t.view(torch.int16).numpy().view(np.uint16) if t.dtype == torch.bfloat16 else t.numpy()
    tens = {n: dev(a) for n, a in stored.items()}
    k(**tens, **kw)
    return {n: host(t) for n, t in tens.items()}


def _check_case(seed, kernels, shape, bh, which=(0, 1), diff_scale=1.0, kappa=KAPPA):
    """Every instance of the kernels ``which`` against the oracle; returns the oracle results."""
    refs = []
    for i in which:
        ir, assigns = kernels[i]
        k = CompiledKernel(ir)
        stored, values = fuzz_inputs(k.fields, ir, shape, seed, diff_scale)
        ref = evaluate(assigns, values, bh)
        march = 'march' in k._emitted and shape[-1] * 2 % 16 == 0
        plain = 'generic' if not march else \
            'march_nomask' if ir.boundary == 'zeros' or ir.ghost_layers == 0 else 'march'
        runs = [(plain, {}), ('generic', dict(_variant='generic'))]
        if march:
            runs.append(('march', dict(_range=ragged_range(shape, ir.ghost_layers))))
        n0 = _launches()
        for instance, kw in runs:
            got = _launch(k, stored, **kw)
            assert k.last_instance == instance, (k.last_instance, instance)
            check_outputs(ir, got, ref, kw.get('_range'), kappa, diff_scale,
                          'seed %d %s %s%s' % (seed, ir.function_name, instance, ' +range' if kw.get('_range') else ''))
        assert _launches() - n0 == len(runs)
        refs += [ref[f.name] for f in ir.output_fields]
    return refs


@pytest.mark.parametrize('seed', range(24))
@pytest.mark.parametrize('dtype', ['float16', 'bfloat16'])
def test_fuzz16_random_stencils(dtype, seed):
    op, kernels, bh, shape = fuzz_case(seed, dtype)
    _check_case(seed, kernels, shape, bh)


@pytest.mark.parametrize('dtype, seed, scale', SCALED)
def test_fuzz16_scaled_gradients(dtype, seed, scale):
    """Adjoints whose upstream gradient is scaled into an edge range: fp16 subnormal results and results beyond 65504
    (stored as inf), bf16 results around fp32's smallest normal and around 1e30."""
    op, kernels, bh, shape = fuzz_case(seed, dtype)
    reached(dtype, scale, _check_case(seed, kernels, shape, bh, which=(1,), diff_scale=scale))


DOUBLE_CASES = [('float16', 6), ('float16', 1), ('bfloat16', 1), ('bfloat16', 6)]
MIXED_SEEDS = [2, 6, 9, 15, 21]


@pytest.mark.parametrize('dtype, seed', DOUBLE_CASES)
def test_fuzz16_data_type_double(dtype, seed):
    """``data_type='double'``: fp64 arithmetic and one rounding from fp64 per stored cell; at κ = 1e-12 a rounding through
    fp32 fails (``DOUBLE_SHAPES``)."""
    shape = DOUBLE_SHAPES[len(fuzz_case(seed, dtype)[3])]
    op, kernels, bh, shape = fuzz_case(seed, dtype, shape=shape, data_type='double')
    assert op.forward_ast_gpu.compute_dtype == np.float64
    _check_case(seed, kernels, shape, bh, which=(0,), kappa=KAPPA_DOUBLE)


@pytest.mark.parametrize('seed', MIXED_SEEDS)
def test_fuzz16_mixed_types(seed):
    """Each field its own type of float16, bfloat16 and float32: the generic kernel, each output checked in its type."""
    op, kernels, bh, shape = fuzz_case(seed, mixed=True)
    _check_case(seed, kernels, shape, bh)
