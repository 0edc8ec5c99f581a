"""GPU: ``bench.py --dump-outputs`` writes what the last timed step computed, and the same arrays from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu

# large enough for the default ('auto') engine to pick the INT8 slicing path, as it does at the headline size
N, D = 400_000, 512
SMALL = ['--n-total', str(N), '--dim', str(D), '--warmup', '1', '--no-e2e', '--no-cpu-baseline', '--no-tf32',
         '--no-configs']


def _bench_dump(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps),
                          '--dump-outputs', str(out_dir)] + SMALL, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith('{')][-1])
    return line, {f: np.load(os.path.join(str(out_dir), f)) for f in sorted(os.listdir(str(out_dir)))}


def test_bench_dump_outputs(tmp_path):
    line1, a = _bench_dump(tmp_path / 'a', 1)
    line2, b = _bench_dump(tmp_path / 'b', 2)
    assert line1['steps'] == 1 and line2['steps'] == 2
    assert line1['config']['engine'] == 'f64_ozaki'
    assert sorted(a) == ['dopt_dhyper_sample.npy', 'hessian_at_opt.npy']
    H, S = a['hessian_at_opt.npy'], a['dopt_dhyper_sample.npy']
    assert H.dtype == S.dtype == np.float64 and H.shape == (D, D) and S.shape == (D, 4096)
    assert sum(os.path.getsize(str(tmp_path / 'a' / f)) for f in a) <= 64 * 10 ** 6
    # the inputs depend only on the arguments: another run (with another number of steps) writes the same arrays
    for f in a:
        np.testing.assert_array_equal(a[f], b[f], err_msg=f)
    # each sampled column is that observation's: H S_j = -r_j x_j is parallel to row j of the seeded design
    from vittles_b200 import ops
    cols = np.sort(np.random.RandomState(20261017).choice(N, 4096, replace=False))
    for k in (0, 1, 2047, 4095):
        x = ops.synth_design(20261017, int(cols[k]), 1, D, torch.device('cuda', 0))[0].cpu().numpy()
        v = H @ S[:, k]
        assert abs(v @ x) / (np.linalg.norm(v) * np.linalg.norm(x)) > 1 - 1e-9, k
