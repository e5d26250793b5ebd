#!/usr/bin/env python
"""Cost of the posterior statistics (sbd_set_posterior) and their diagnostics (sbd_set_posterior_diagnostics) in the
SAPG main loop.

For each configuration the same seeded problem is run with the statistics off, with post_mean only, with
post_levels L = 1 and L = 4, and with L = 4 plus the diagnostics at the automatic batch length, alternating the variants; each variant reports the best of --reps runs of the
device-timed main loop (sbd_traces.seconds_main) as chain-steps/s.  The runs go through sbd_sapg_run_dev with y in
HBM and no trace or sample copies, so only the main loop is timed.  The card's name, power limit and max SM clock
are printed with the numbers.

  python tools/posterior_overhead.py [--reps 3] [--out results.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (rows, cols, chains, use_graph, main-loop steps)
CONFIGS = [(4096, 4096, 8, 0, 12), (2160, 3840, 8, 0, 12), (512, 512, 1, 0, 200), (256, 256, 1, 1, 400)]
# (name, post_mean, post_levels, post_batch)
VARIANTS = [("off", 0, 0, 0), ("post_mean", 1, 0, 0), ("L1", 0, 1, 0), ("L4", 0, 4, 0), ("L4_diag", 0, 4, -1)]


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def params(H, rows, cols, nch, steps, use_graph, post_mean):
    sig2 = 4.0
    op = dict(samples=steps + 1, warmup=3, burnIn=1, psf_size=7, phi=0.0, min_th=1e-3, max_th=1.0, th_init=0.01,
              w1_init=0.5, w2_init=0.3, min_w1=0.1, max_w1=1.0, min_w2=0.1, max_w2=1.0, w1=0.4, w2=0.3,
              fix_w1=0, fix_w2=0, fix_sigma=0, d_exp=0.8, d_scale=1.0, sigma_init=sig2, sigma_min=0.5 * sig2,
              sigma_max=2 * sig2, use_graph=use_graph)
    Lf = 0.993 ** 2 / op["sigma_max"]
    op["lambda"] = min(5 / Lf, 2.0)
    op["gamma"] = 0.98 / (Lf + 1 / op["lambda"])
    c = dict(sigma=1000.0, theta=0.01, w1=10.0, w2=10.0, lam=1.0, gam=1.0)
    return H.make_params(H.GAUSSIAN, op, c, n_chains=nch, seed=11, post_mean=post_mean)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--configs", default="all", help="comma-separated indices into CONFIGS, or 'all'")
    a = ap.parse_args()
    import torch
    import sbd_b200
    from sbd_b200 import host as H
    from sbd_b200._lib import lib, sbd_traces
    info = gpu_info()
    print("GPU (name, power limit, max SM clock):", info, flush=True)
    sel = range(len(CONFIGS)) if a.configs == "all" else [int(i) for i in a.configs.split(",")]
    rows_out = []
    for ci in sel:
        rows, cols, nch, use_graph, steps = CONFIGS[ci]
        eng = sbd_b200.Engine(rows, cols, 7, H.GAUSSIAN, 0.0, max_batch=nch)
        g = torch.Generator(device="cpu").manual_seed(ci)
        y = (128 + 40 * torch.randn(cols, rows, generator=g, dtype=torch.float64)).abs().cuda()   # column-major image
        best = {v[0]: 0.0 for v in VARIANTS}
        for rep in range(a.reps + 1):                    # rep 0 warms every variant up (allocations, graphs)
            for name, pm, L, b in VARIANTS:
                prm = params(H, rows, cols, nch, steps, use_graph, pm)
                tr = sbd_traces()
                eng._check(lib.sbd_set_posterior(eng._h, L))
                eng._check(lib.sbd_set_posterior_diagnostics(eng._h, b))
                eng._check(lib.sbd_sapg_run_dev(eng._h, C.c_void_p(y.data_ptr()), None, C.byref(prm), C.byref(tr)))
                eng._check(lib.sbd_set_posterior_diagnostics(eng._h, 0))
                eng._check(lib.sbd_set_posterior(eng._h, 0))
                rate = steps * nch / tr.seconds_main
                if rep > 0:
                    best[name] = max(best[name], rate)
        row = dict(rows=rows, cols=cols, chains=nch, use_graph=use_graph, steps=steps, gpu=info,
                   **{f"chain_steps_per_s_{k}": v for k, v in best.items()})
        row["overhead_L1_vs_post_mean"] = best["post_mean"] / best["L1"] - 1
        row["overhead_L4_vs_post_mean"] = best["post_mean"] / best["L4"] - 1
        row["overhead_L4_diag_vs_L4"] = best["L4"] / best["L4_diag"] - 1
        print(json.dumps(row), flush=True)
        rows_out.append(row)
        eng.close()
        del y
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(rows_out, f, indent=1)


if __name__ == "__main__":
    main()
