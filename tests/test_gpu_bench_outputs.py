"""bench.py --dump-outputs: what the timed steps computed, written so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
           "--no-cpu", "--no-sharded", "--dump-outputs", str(out_dir)]
    p = subprocess.run(cmd, cwd=out_dir.parent, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    line, a = run_bench(tmp_path / "a", 3)
    assert line["steps"] == 3
    assert {"losses", "alpha", "log_alpha", "priorities", "policy.fc1.weight", "q1.fc4.bias", "q2_target.fc1.weight"} <= set(a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert np.isfinite(a["losses"]).all() and a["priorities"].shape == (1_000_000,)
    _, b = run_bench(tmp_path / "b", 3)      # same arguments: same seeded inputs, same outputs
    assert a.keys() == b.keys()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    line, c = run_bench(tmp_path / "c", 4)   # one more timed step: one more update behind the outputs
    assert line["steps"] == 4
    assert not np.array_equal(a["losses"], c["losses"]) and not np.array_equal(a["policy.fc1.weight"], c["policy.fc1.weight"])
