"""CPU checks of bench.py: the reference arm (the oracle timed on the host cores) runs REAL iterations at --size and
prints the JSON line of the contract; under a multi-rank launch only rank 0 works."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_line():
    lines = run(["--impl", "reference", "--size", "256", "--steps", "3", "--warmup", "1"])
    assert len(lines) == 1
    d = lines[0]
    assert d["impl"] == "reference" and d["steps"] == 3 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["unit"] == "chain-steps/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["config"]["image"] == "256x256" and d["config"]["total_chains"] == 64 and d["scaling"] == "strong"
    # value = 1 / (mean seconds per real iteration); no extrapolation factor anywhere
    assert abs(d["value"] * d["ms_per_step"] / 1e3 - 1.0) < 1e-9
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "no extrapolation" in cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None


def test_reference_arm_other_ranks_do_nothing():
    lines = run(["--impl", "reference", "--size", "256", "--steps", "2", "--warmup", "1", "--gpus", "2"],
                env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert lines == []


def test_chain_split_is_strong_scaling():
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    a = argparse.Namespace(total_chains=64, chains_per_gpu=0, size=4096)
    assert [bench.chains_for(a, w) for w in (1, 2, 4, 8)] == [(64, 64), (32, 64), (16, 64), (8, 64)]
    assert bench.scaling_kind(a) == "strong"
    a.chains_per_gpu = 8
    assert bench.chains_for(a, 4) == (8, 32) and bench.scaling_kind(a) == "weak"
    assert bench.alg_bytes_per_chain_step(4096 * 4096) == 1144 * 4096 * 4096
    assert bench.chamb_plan_n4(25) == 4 and bench.chamb_plan_n4(20) == 4


def test_dump_sample_is_fixed_and_bounded():
    """--dump-outputs keeps the chains' last samples at seeded pixels: the same for every run, within 32 MiB (float64)
    with the index row, and every pixel when the image is small."""
    sys.path.insert(0, ROOT)
    import bench
    for npix, nch in ((4096 * 4096, 64), (4096 * 4096, 1), (2048 * 2048, 8)):
        idx = bench.last_sample_pixels(npix, nch)
        assert np.array_equal(idx, bench.last_sample_pixels(npix, nch))
        assert idx[0] >= 0 and idx[-1] < npix and np.all(np.diff(idx) > 0)
        assert (nch + 1) * idx.size * 8 <= 32 << 20
    assert np.array_equal(bench.last_sample_pixels(256 * 256, 8), np.arange(256 * 256))


def test_dump_outputs_is_for_the_gpu_arm():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
