"""bench.py without a GPU: the --dump-outputs writer and the arguments bench.py refuses."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_types_budget_and_fixed_sample(tmp_path, monkeypatch):
    limit = 8192
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', limit)
    arrays = {'big': torch.arange(10000, dtype=torch.float32), 'small': torch.ones(3, 2, dtype=torch.bfloat16), 'loss': 0.25}
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {d: {k: np.load(tmp_path / d / (k + '.npy')) for k in arrays} for d in ('a', 'b')}
    a = got['a']
    assert a['small'].dtype == np.float32 and a['small'].shape == (3, 2) and (a['small'] == 1).all()
    assert a['loss'].dtype == np.float64 and a['loss'] == 0.25
    # the large array is sampled down to what the small ones leave of the budget, counted in file bytes
    files = sum(f.stat().st_size for f in (tmp_path / 'a').iterdir())
    assert a['big'].dtype == np.float32 and a['big'].size < 10000 and limit - 4 < files <= limit
    assert (np.diff(a['big']) > 0).all()                                          # distinct elements, in their original order
    for k in arrays:
        assert np.array_equal(a[k], got['b'][k]), k


@pytest.mark.parametrize('argv', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'out']])
def test_bench_refuses_bad_arguments(tmp_path, argv):
    res = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + argv, capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    assert res.returncode == 2, res.stderr[-2000:]
    assert os.listdir(tmp_path) == []
