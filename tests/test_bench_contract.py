"""bench.py's JSON contract (reference arm runs on CPU; the GPU arm is covered by the `gpu` marker)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
             'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches'}


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '2',
                          '--warmup', '1', '--workload', 'c2', '--shape', '512', '512'],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert BASE_KEYS <= set(line)
    assert line['impl'] == 'reference' and line['unit'] == 'Mcell-updates/s' and line['value'] > 0
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1
    assert line['e2e'] == {'value': line['value'], 'unit': line['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in line['config'] and line['vs_baseline'] is None


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2'],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ''


@pytest.mark.parametrize('argv, message', [(['--steps', '0'], '--steps must be at least 1'),
                                            (['--impl', 'reference', '--dump-outputs', 'x'], 'needs --impl ours')])
def test_bad_arguments_are_refused(argv, message):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + argv,
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and message in out.stderr


@pytest.mark.gpu
@pytest.mark.no_launch          # the launches happen in the bench.py process this test starts
def test_gpu_arm_line_small(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '3', '--warmup', '3',
                          '--workload', 'c3', '--shape', '128', '128', '256', '--e2e-steps', '1', '--no-cpu-baseline',
                          '--dump-outputs', str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert BASE_KEYS | {'roofline', 'clocks'} <= set(line)
    assert line['gpu_launches'] == 6
    assert line['roofline']['bound'] == 'hbm' and 0 < line['roofline']['frac'] < 1.5
    assert line['e2e']['h2d_bytes_per_step'] == 2 * 128 * 128 * 256 * 4
    assert line['config']['kernel_variants'] == {'forward': 'march', 'adjoint': 'march'}
    # small enough to be written whole: the forward output and the input gradient, as the timed step computed them from
    # bench.py's seeded inputs (regenerated here the same way) — checked against the numpy oracle
    import torch
    from oracle import forward_backward
    from pystencils_autodiff_b200.configs import make_config
    from pystencils_autodiff_b200.datahandling import SlabStencilOp
    assert sorted(os.listdir(tmp_path)) == ['diffu.npy', 'out.npy']
    shape = (128, 128, 256)
    op = make_config('c3', shape=shape, boundary_handling='zeros')
    slab = SlabStencilOp(op, local_shape=shape, device=torch.device('cuda', 0))
    g = torch.Generator(device='cuda:0')
    g.manual_seed(1234)
    slab.randomize(g)
    ref_out, ref_din = forward_backward(op, {'u': slab.dh.owned('u').cpu().numpy()},
                                        {'out': slab.dh.owned('diffout').cpu().numpy()})
    for name, ref in (('out', ref_out['out']), ('diffu', ref_din['diffu'])):
        a = np.load(os.path.join(tmp_path, name + '.npy'))
        assert a.shape == shape and a.dtype == np.float32
        assert np.abs(a - ref).max() / np.abs(ref).max() <= 1e-6, name


@pytest.mark.gpu
@pytest.mark.no_launch
def test_gpu_arm_dumps_the_same_sample_every_run(tmp_path):
    """Outputs over the size limit are sampled at fixed indices, and the inputs are seeded: two runs dump the same values."""
    dumps = []
    for run in ('a', 'b'):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '2', '--warmup', '1',
                              '--workload', 'c2', '--shape', '4096', '4096', '--only-headline', '--no-e2e',
                              '--no-cpu-baseline', '--dump-outputs', str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr
        assert json.loads(out.stdout.strip().splitlines()[-1])['steps'] == 2
        assert sorted(os.listdir(tmp_path / run)) == ['diffu.npy', 'out.npy']
        dumps.append({n: np.load(str(tmp_path / run / (n + '.npy'))) for n in ('diffu', 'out')})
    assert sum(os.path.getsize(str(tmp_path / 'a' / (n + '.npy'))) for n in ('diffu', 'out')) <= 64 * 10**6
    for n in ('diffu', 'out'):
        assert dumps[0][n].dtype == np.float32 and dumps[0][n].ndim == 1 and 10**6 < dumps[0][n].size < 4096 * 4096
        assert np.array_equal(dumps[0][n], dumps[1][n])
