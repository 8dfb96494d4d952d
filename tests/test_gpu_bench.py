"""bench.py --dump-outputs on the device: the same arguments give the same outputs, and --steps sets which step they are from
(config 3: the eager loop; config 2: the CUDA-graph replays its headline is quoted on)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(config, steps, out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", str(config), "--envs-per-gpu", "256", "--steps", str(steps),
                        "--warmup", "3", "--no-cpu-baseline", "--no-e2e", "--no-fill-context", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


@pytest.mark.parametrize("config", [3, 2])
def test_bench_dump_outputs_repeat_and_follow_steps(config, tmp_path):
    a, b, c = _bench(config, 5, tmp_path / "a"), _bench(config, 5, tmp_path / "b"), _bench(config, 10, tmp_path / "c")
    assert {"obs", "reward", "terminated", "truncated", "info_cte", "info_position"} <= set(a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64_000_000
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a), [k for k in a if not np.array_equal(a[k], b[k])]
    assert a["obs"].any() and not np.array_equal(a["info_position"], c["info_position"])   # five more steps moved the cars
