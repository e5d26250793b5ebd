#!/usr/bin/env python
"""FFT operators and SAPG at image sizes that are not powers of two (mixed-radix path, fft_any.cuh) next to their
power-of-two neighbours.  The card's name and power limit are printed first and belong to every number below them.

    python tools/fft_any_sweep.py [--out DIR] [--steps 20]

1. A / A' per call, batch 8: host clock around 10 calls that ends in a device synchronise (so it includes the launch
   cost and the per-call PSF refresh), in algorithmic bytes per second (64 * P bytes per image, DESIGN.md section 4).
2. SAPG main-loop chain-steps/s (Gaussian PSF, the bench configuration; CUDA events of the library, sbd_traces
   seconds_main) and the phase split of sbd_phase_times (a second, profiled run: profiling serialises the two streams
   of an iteration): 2160x3840 x 8 chains vs 2048x4096 x 8, and 480x640 x 1 chain vs 512x512 x 1.
3. Device time of every FFT kernel of a SAPG run (torch.profiler, CUDA activity) at 2160x3840 x 8 and 2048x4096 x 8,
   with the bytes each kernel must move (16 P per image: 8 P in, 8 P out) over its time.
One JSON line per measurement; with --out also written to DIR/fft_any_sweep.jsonl.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OP_SIZES = [(480, 640), (512, 512), (1000, 1000), (1024, 1024), (1080, 1920), (2048, 2048), (2160, 3840), (2048, 4096),
            (3000, 4000), (4096, 4096)]
SAPG_CASES = [((2160, 3840), 8), ((2048, 4096), 8), ((480, 640), 1), ((512, 512), 1)]


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20, help="SAPG main-loop iterations")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    import bench as B
    import sbd_b200
    from sbd_b200 import host as H
    from sbd_b200._lib import lib
    if not torch.cuda.is_available():
        sys.exit("fft_any_sweep: needs a GPU (no CPU numbers)")
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    emit({"card": card(), "torch_device": torch.cuda.get_device_name(0)})

    # ---- 1. A / A' throughput, batch 8
    batch = 8
    for rows, cols in OP_SIZES:
        npix = rows * cols
        eng = sbd_b200.Engine(rows, cols, 7, H.GAUSSIAN, 0.0, batch, 0)
        x = torch.rand(batch, cols, rows, dtype=torch.float64, device="cuda") * 255.0
        out = torch.empty_like(x)
        psi = (C.c_double * 2)(0.4, 0.3)
        res = {"op_size": [rows, cols], "batch": batch, "path": "pow2" if (rows & (rows - 1)) == 0 and (cols & (cols - 1)) == 0 else "mixed-radix"}
        for name, opsel in (("A", 0), ("AT", 1)):
            def run():
                rc = lib.sbd_blur_dev(eng._h, x.data_ptr(), psi, opsel, out.data_ptr(), batch)
                assert rc == 0, lib.sbd_last_error(eng._h)
            for _ in range(3):
                run()
            lib.sbd_synchronize(eng._h)
            best = 1e30
            for _ in range(a.reps):
                lib.sbd_synchronize(eng._h)
                t0 = time.perf_counter()
                for _ in range(10):
                    run()
                lib.sbd_synchronize(eng._h)                 # the library runs on its own stream
                best = min(best, (time.perf_counter() - t0) * 1e3 / 10)
            res[name] = {"ms_per_call": best, "alg_GBps": 64.0 * npix * batch / (best * 1e-3) / 1e9,
                         "ns_per_pixel": best * 1e6 / (npix * batch)}
        emit(res)
        eng.close()
        del x, out
        torch.cuda.empty_cache()

    # ---- 2. SAPG main loop
    for (rows, cols), nch in SAPG_CASES:
        npix = rows * cols
        eng = sbd_b200.Engine(rows, cols, 7, H.GAUSSIAN, 0.0, nch, 0)
        cm = np.load(os.path.join(ROOT, "tests", "golden", "cman_u8.npy")).astype(np.float64)
        x_true = np.tile(cm, ((rows + 255) // 256, (cols + 255) // 256))[:rows, :cols].copy()
        Ax = eng.blur(x_true, B.PSI_TRUE, H.OP_A)
        nrm = float(np.linalg.norm(Ax - Ax.mean()))
        sig = lambda b: nrm / np.sqrt(npix * 10 ** (b / 10))
        y = Ax + sig(30) * np.random.default_rng(2).standard_normal((rows, cols))
        op, c = B.gaussian_op(rows, sig(30), sig(15), sig(45), 0.993, a.steps + 1, 3)
        prm = H.make_params(H.GAUSSIAN, op, c, n_chains=nch, seed=1, chain_offset=0, total_chains=nch)
        eng.sapg(y, prm, want_X_warm=False)                             # warm-up run (modules, graphs)
        best = 1e30
        for _ in range(3):
            o = eng.sapg(y, prm, want_X_warm=False)
            best = min(best, o["seconds_main"])
        rate = a.steps * nch / best
        eng.set_profile(True)
        eng.sapg(y, prm, want_X_warm=False)
        eng.set_profile(False)
        ph = {k: v[0] / a.steps for k, v in eng.phase_times().items()}
        fft_ms = ph["spectral_inverse"] + ph["spectral_forward"]
        emit({"sapg_size": [rows, cols], "chains": nch, "steps": a.steps, "chain_steps_per_s": rate,
              "ms_per_step": best * 1e3 / a.steps, "ns_per_pixel_step": best * 1e9 / a.steps / (npix * nch),
              "phase_ms_per_step_profiled": ph, "fft_ns_per_pixel_step_profiled": fft_ms * 1e6 / (npix * nch)})
        eng.close()
        torch.cuda.empty_cache()

    # ---- 3. device time per FFT kernel inside SAPG
    from torch.profiler import profile, ProfilerActivity
    for (rows, cols), nch in SAPG_CASES[:2]:
        npix = rows * cols
        eng = sbd_b200.Engine(rows, cols, 7, H.GAUSSIAN, 0.0, nch, 0)
        y = np.random.default_rng(3).uniform(0, 255, (rows, cols))
        op, c = B.gaussian_op(rows, 5.0, 2.0, 10.0, 0.993, 6, 3)
        prm = H.make_params(H.GAUSSIAN, op, c, n_chains=nch, seed=1, chain_offset=0, total_chains=nch)
        prm.use_graph = 0
        eng.set_option("overlap", 0)                        # one stream: no kernel shares the SMs with the one timed
        eng.sapg(y, prm, want_X_warm=False)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.sapg(y, prm, want_X_warm=False)
            torch.cuda.synchronize()
        durs = {}
        for e in prof.events():                             # kernel events: the CPU side is cudaLaunchKernel
            if "k_rows" in e.name or "k_cols" in e.name:
                durs.setdefault(e.name.split("(")[0].replace("void ", ""), []).append(e.time_range.elapsed_us())
        kern = {}
        for k, d in durs.items():
            # the median skips the single one-image call (rows pass / COL_FWD of y) of a kernel the steps use on all chains
            imgs = 1 if len(d) == 1 else nch
            us = float(np.median(d))
            kern[k] = {"calls": len(d), "images": imgs, "us_median": us, "GBps_16P": 16.0 * npix * imgs / (us * 1e-6) / 1e9}
        emit({"kernels_size": [rows, cols], "chains": nch, "kernels": kern})
        eng.close()
        torch.cuda.empty_cache()

    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "fft_any_sweep.jsonl"), "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
