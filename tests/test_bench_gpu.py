"""bench.py on the GPU: --dump-outputs writes what the last timed step of the default workload computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    out = tmp_path / 'dump'
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '2', '--warmup', '3', '--no-extras', '--dump-outputs', str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line['steps'] == 2
    depth = np.load(out / 'output_depth.npy')
    assert depth.dtype == np.float32 and depth.shape == (1, 1, 352, 1216) and np.isfinite(depth).all()
    params = np.load(out / 'adapted_parameters.npy')
    assert params.dtype == np.float32 and params.ndim == 1 and params.size > 0 and np.isfinite(params).all()
    for k, v in line['last_losses'].items():           # the losses the bench line reports are the dumped step's
        assert np.load(out / (k + '.npy')) == v, k
    assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
