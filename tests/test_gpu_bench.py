"""bench.py --dump-outputs on the GPU: two runs with the same arguments write the same arrays (names, shapes, and values
up to the order in which the backward's float atomics add up), as float32 / float64 and within 64 MB in all, and the
JSON line reports the number of timed steps asked for."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.util import rel_linf

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1", "--no-variants",
           "--no-kernels", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3
    files = sorted(os.listdir(out_dir))
    assert files and all(f.endswith(".npy") for f in files)
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in files) <= 64 << 20
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in files}


def test_bench_dump_outputs_repeat(tmp_path):
    a, b = _bench_dump(tmp_path / "a"), _bench_dump(tmp_path / "b")
    assert a.keys() == b.keys()
    assert "loss" in a and "input_grad" in a and sum(k.startswith("grad.") for k in a) > 100
    assert float(a["loss"]) > 0
    worst = {}
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and a[k].shape == b[k].shape, k
        assert np.isfinite(a[k]).all(), k
        worst[k] = rel_linf(torch.from_numpy(a[k]), torch.from_numpy(b[k]))
    print("largest run-to-run differences", sorted(worst.items(), key=lambda kv: -kv[1])[:5])
    # the prompt-token gradients, summed over all windows by float atomics, move by ~1e-3 between runs (B200, 20 steps);
    # a different input, weight or dropout seed moves every array by O(1)
    assert max(worst.values()) < 2e-2, worst
