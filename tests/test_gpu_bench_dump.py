"""bench.py --dump-outputs: two runs with the same arguments write the same arrays (float64, within 64 MB), the
trajectories have one entry per timed step plus the initial one, and the JSON line reports the --steps it was given."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return lines[0]


def test_dump_outputs_are_reproducible(tmp_path):
    steps, chains, n = 6, 8, 256
    args = ["--size", str(n), "--total-chains", str(chains), "--steps", str(steps), "--warmup", "3",
            "--no-extras", "--no-size-sweep", "--no-cpu-baseline"]
    dumps = []
    for d in ("a", "b"):
        line = run(args + ["--dump-outputs", str(tmp_path / d)])
        assert line["steps"] == steps
        dumps.append({f[:-4]: np.load(tmp_path / d / f) for f in sorted(os.listdir(tmp_path / d))})
    a, b = dumps
    assert sorted(a) == sorted(b)
    assert {"thetas", "sigmas", "psi0", "psi1", "chambolle_iters", "X_last_sample", "X_last_sample_index"} <= set(a)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
    assert a["thetas"].shape == (steps + 1,) and np.all(np.isfinite(a["thetas"]))
    idx = a["X_last_sample_index"]
    assert a["X_last_sample"].shape == (chains, idx.size) and np.all(np.isfinite(a["X_last_sample"]))
    assert idx.min() >= 0 and idx.max() < n * n and np.all(np.diff(idx) > 0)
