"""bench.py's contract: the reference arm's JSON line, that the GPU arm refuses to run without a device instead of
falling back to anything, and --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, gpu=False):
    env = dict(os.environ) if gpu else dict(os.environ, CUDA_VISIBLE_DEVICES='')
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + list(args), capture_output=True, text=True,
                          env=env, timeout=900, cwd=ROOT)


def test_reference_arm_json_line():
    r = _run('--impl', 'reference', '--steps', '1', '--warmup', '1')
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'images/s' and d['higher_is_better'] is True
    assert d['metric'].startswith('x4 SR images/sec') and d['n_gpus'] == 1 and d['steps'] == 1
    assert d['value'] > 0 and abs(d['ms_per_step'] * d['value'] / 1e3 - 2) < 1e-6          # two images per step
    assert d['vs_baseline'] is None and d['data'] == 'synthetic' and 'workload' in d['config']
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] == (os.cpu_count() or 1) and cb['value'] == d['value'] and cb['sample']
    assert d['e2e'] == {'value': d['value'], 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_gpu_arm_fails_loudly_without_a_device():
    r = _run('--steps', '1')
    assert r.returncode != 0
    assert 'no CUDA device' in (r.stderr + r.stdout) and 'no CPU fallback' in (r.stderr + r.stdout)


def _documented_dump(k, t):
    """What dump_outputs' docstring promises for the k-th output `t`: the whole array, or the values at sorted flat
    (logical NCHW) positions drawn from torch.Generator().manual_seed(k) when it exceeds its share of DUMP_BYTES."""
    import bench
    dt = torch.float32 if t.is_floating_point() else torch.float64
    n = bench.DUMP_BYTES // len(bench.OUTPUT_NAMES) // dt.itemsize
    if t.numel() > n:
        pos = torch.randint(t.numel(), (n,), generator=torch.Generator().manual_seed(k)).sort().values
        t = t.flatten()[pos.to(t.device)]
    return t.to(dt).cpu().numpy()


def test_dump_outputs_names_dtypes_and_fixed_sample(tmp_path):
    import bench
    g = torch.Generator().manual_seed(0)
    small = [torch.randint(0, 1444, (4, 38, 38), generator=g), torch.rand(4, 38, 38, generator=g)]
    big = [torch.randn(3, 64, 160, 160, generator=g).contiguous(memory_format=torch.channels_last) for _ in range(6)]
    bench.dump_outputs(small + big, str(tmp_path))
    files = sorted(os.listdir(tmp_path))
    assert files == sorted(n + '.npy' for n in bench.OUTPUT_NAMES)
    assert sum(os.path.getsize(tmp_path / f) for f in files) < 64e6
    for k, (name, t) in enumerate(zip(bench.OUTPUT_NAMES, small + big)):
        a, want = np.load(tmp_path / (name + '.npy')), _documented_dump(k, t)
        assert a.dtype == want.dtype == (np.float64 if k == 0 else np.float32) and np.array_equal(a, want), name
        assert a.shape == (t.shape if k < 2 else (bench.DUMP_BYTES // 8 // 4,)), name


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_step_outputs(tmp_path):
    """--steps sets the number of timed steps (the library's launch count in the timed region scales with it), and the
    dump holds what hot_path_step computes on the same seeded inputs, at the documented positions."""
    import bench
    import mrefsr_b200 as M
    runs = {}
    for steps in (2, 3):
        r = _run('--batch', '1', '--refs', '2', '--steps', str(steps), '--warmup', '1', '--no-e2e', '--no-cpu-baseline',
                 '--no-full-model', '--no-extras', '--dump-outputs', str(tmp_path / str(steps)), gpu=True)
        assert r.returncode == 0, r.stderr[-2000:]
        runs[steps] = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('{')][-1])
        assert runs[steps]['steps'] == steps
    assert runs[2]['gpu_launches'] > 0 and runs[3]['gpu_launches'] * 2 == runs[2]['gpu_launches'] * 3
    outs = bench.hot_path_step(M, bench.make_inputs(1, 2, 1234, 'cuda:0'), 1, 2, 'auto', 'auto')
    for k, (name, t) in enumerate(zip(bench.OUTPUT_NAMES, outs, strict=True)):
        want = _documented_dump(k, t)
        for steps in (2, 3):
            a = np.load(tmp_path / str(steps) / (name + '.npy'))
            assert a.dtype == want.dtype and a.shape == want.shape, (name, steps)
            np.testing.assert_allclose(a, want, rtol=1e-5, atol=1e-6, err_msg='%s, --steps %d' % (name, steps))
