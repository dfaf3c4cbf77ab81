"""bench.py contract pieces that run without a GPU: the reference arm (`--impl reference`, CPU oracle port) prints ONE JSON
line with the keys the driver reads, non-zero ranks print nothing, and the product arm refuses to run without CUDA
(no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args, capture_output=True, text=True,
                          timeout=timeout, env=e, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    r = _run(['--impl', 'reference', '--tiny', '--steps', '1', '--warmup', '1'])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    out = json.loads(lines[0])
    assert out['impl'] == 'reference' and out['higher_is_better'] is True and out['unit'] == 'denoise_steps/s'
    assert out['value'] > 0 and out['steps'] == 1
    for k in ('metric', 'n_gpus', 'warmup', 'ms_per_step', 'scaling', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in out, k
    assert out['cpu_baseline']['kind'] == 'port' and out['cpu_baseline']['cores'] >= 1
    assert out['e2e']['h2d_bytes_per_step'] == 0 and out['e2e']['d2h_bytes_per_step'] == 0
    assert 'workload' in out['config'] and 'model' not in out['config']


def test_reference_arm_nonzero_rank_is_silent():
    r = _run(['--impl', 'reference', '--tiny', '--steps', '1', '--warmup', '1', '--gpus', '2'],
             env={'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_product_arm_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    r = _run(['--tiny', '--steps', '1', '--warmup', '1'])
    assert r.returncode != 0 and 'needs a GPU' in (r.stderr + r.stdout)


def test_product_code_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the package may import it, and bench.py may do so only inside the
    two CPU-baseline functions."""
    import re
    pkg = os.path.join(ROOT, 'mix-of-show_b200')
    pat = re.compile(r'^\s*(from\s+oracle\b|import\s+oracle\b)', re.M)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert not pat.search(src), f'{os.path.join(dirpath, f)} imports oracle'
    src = open(os.path.join(ROOT, 'bench.py')).read()
    allowed = ('def build_cpu_reference', 'def cpu_reference_steps')
    for m in pat.finditer(src):
        head = src[:m.start()]
        last_def = head.rfind('\ndef ')
        assert src[last_def + 1:].startswith(allowed), 'bench.py imports oracle outside the CPU-baseline functions'


def test_dump_outputs_writes_float32_within_budget(tmp_path, monkeypatch):
    """An array over its share of the budget is replaced by the same seeded sample of its elements every time."""
    import numpy as np
    import torch

    import bench
    monkeypatch.setattr(bench, 'DUMP_BYTES', 4096)
    big = torch.arange(5000, dtype=torch.float64).view(50, 100)
    small = torch.ones(2, 3, dtype=torch.float16)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'big': big, 'small': small})
    a, b = np.load(tmp_path / 'a' / 'big.npy'), np.load(tmp_path / 'b' / 'big.npy')
    assert a.dtype == np.float32 and a.shape == (512,) and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and np.all(np.isin(a, big.numpy()))
    s = np.load(tmp_path / 'a' / 'small.npy')
    assert s.dtype == np.float32 and s.shape == (2, 3) and np.all(s == 1)


@pytest.mark.gpu
def test_product_arm_dumps_its_outputs(cuda, tmp_path):
    import numpy as np
    r = _run(['--tiny', '--steps', '2', '--warmup', '1', '--no-train', '--no-cpu-baseline', '--dump-outputs', str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])['steps'] == 2
    shapes = {'latents': (1, 4, 64, 64), 'eps': (2, 4, 64, 64), 'e2e_latents': (1, 4, 64, 64)}
    assert sorted(os.listdir(tmp_path)) == sorted(n + '.npy' for n in shapes)
    for n, shape in shapes.items():
        a = np.load(tmp_path / (n + '.npy'))
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all(), n
