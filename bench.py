#!/usr/bin/env python
"""bench.py - MYULA (SAPG main-loop) iterations per second on B200.

  python bench.py --gpus N --steps K --warmup W [--impl reference]

Workload (BASELINE.json configs[3], the one the headline metric is quoted on):
synthetic 4096x4096 Gaussian-PSF SAPG with 64 MYULA chains sharded over the N
GPUs (64 / 32 / 16 / 8 chains per GPU at N = 1 / 2 / 4 / 8: strong scaling,
SURVEY.md 8e), NCCL all-gather of the per-chain stochastic gradients at every
outer iteration.  A "step" is one SAPG main-loop iteration of every chain
(SAPG_algorithm_Guassian.m:158-248: Langevin update, Chambolle prox with 25
sweeps, spectral gradients, theta / sigma^2 / w1 / w2 updates).  W warm-up steps
are real MYULA warm-up iterations (Guassian.m:78-91) and are not timed.
`--chains-per-gpu n` switches to weak scaling with n chains on every GPU.

  value : chain-steps/s with y and X0 resident in HBM (device-timed main loop)
  e2e   : same metric through the host-pointer C ABI (sbd_sapg_run): y copied
          from pinned host memory and trajectories + last samples copied back,
          inside the timed region (wall clock around the call)
  --impl reference : the CPU restatement of the reference (oracle/, numpy +
          scipy.fft on all host cores + the plain-C TV prox) timed on REAL
          iterations at --size: one chain, K steps after W warm-up steps.
  --dump-outputs DIR : after the timed steps, writes what the device-timed main
          loop returned (its trajectories and a seeded sample of every chain's
          last sample) as DIR/<name>.npy in float64, so that two builds can be
          compared output for output on identical inputs.

At N = 1 the line also carries (extra keys) the other BASELINE.json configs:
configs[0] the full run_Gaussian_demo.m run on cameraman 256^2, configs[1]
Moffat on boat 512^2, configs[4] the operator sweep; at N > 1 configs[2]
(Laplace SAPG, one images/*.png per GPU, replicas without a collective).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PSI_TRUE = (0.4, 0.3)            # run_Gaussian_demo.m:78-79
PSI_INIT = (0.5, 0.3)            # run_Gaussian_demo.m:68-69 (estimating the bandwidths, Q17)
CHAMBOLLE_K = 25                 # run_Gaussian_demo.m:188
EVMAX = 0.993                    # evMax of A'A at (w1,w2)=(1,1): what the reference's power iteration returns
UNIT = "chain-steps/s"
METRIC = "MYULA chain-iterations/sec"
# --dump-outputs: trajectories of the timed main loop besides thetas / sigmas / chambolle_iters, and how many values of
# the chains' last samples are kept (all chains of the rank and the pixel indices together: 32 MiB in float64)
DUMP_TRACES = ("psi0", "psi1", "grad_theta", "grad_psi0", "grad_psi1", "grad_sigma", "logPiTraceX", "gXTrace")
DUMP_LAST_SAMPLE_VALUES = 1 << 22
DUMP_SEED = 0


def alg_bytes_per_chain_step(npix, k=CHAMBOLLE_K):
    """SURVEY.md 8(d): B_alg = (144 + 40 K) * P bytes per chain per main-loop step."""
    return (144 + 40 * k) * npix


def golden(name):
    return os.path.join(ROOT, "tests", "golden", name)


def synthetic_truth(n):
    """cman (256x256) periodically tiled to n x n (SURVEY.md 8d)."""
    cm = np.load(golden("cman_u8.npy")).astype(np.float64)
    reps = (n + 255) // 256
    return np.tile(cm, (reps, reps))[:n, :n].copy()


def last_sample_pixels(npix, nch, seed=DUMP_SEED):
    """Sorted pixel indices (column-major, as the device holds an image) at which --dump-outputs keeps every chain's
    last sample: a fixed, seeded choice that depends on the image size and the number of chains only."""
    per = max(1, min(npix, DUMP_LAST_SAMPLE_VALUES // (nch + 1)))        # nch rows of values + the index row
    return np.sort(np.random.default_rng(seed).choice(npix, per, replace=False))


def write_dump(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def gaussian_op(n, sigma, sigma_min, sigma_max, evMax, samples, warmup):
    """op / c of run_Gaussian_demo.m:34-85,177-191 with fix_w1 = fix_w2 = 0."""
    op = dict(samples=samples, warmup=warmup, burnIn=max(2, (samples * 80) // 100), psf_size=7, phi=0.0,
              min_th=1e-3, max_th=1.0, min_w1=0.1, max_w1=1.0, min_w2=0.1, max_w2=1.0,
              th_init=0.01, w1_init=PSI_INIT[0], w2_init=PSI_INIT[1], w1=PSI_TRUE[0], w2=PSI_TRUE[1],
              fix_w1=0, fix_w2=0, fix_sigma=0, d_exp=0.8, d_scale=0.01 / 0.01,
              sigma=sigma, sigma_init=(sigma_min ** 2 + sigma_max ** 2) / 2,
              sigma_min=sigma_min ** 2, sigma_max=sigma_max ** 2, chambolleit=CHAMBOLLE_K)
    Lf = min(evMax ** 2 / sigma_min ** 2, evMax ** 2 / sigma_max ** 2)
    op["lambda"] = min(5 / Lf, 2.0)
    op["gamma"] = 0.98 / (Lf + 1 / op["lambda"])
    c = dict(sigma=1000.0, theta=0.01, w1=10.0, w2=10.0, lam=1.0, gam=1.0)
    return op, c


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [s.strip() for s in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            # the busiest half of the samples = "under load"
            top = sorted(sm)[len(sm) // 2:]
            out = {"sm_mhz": float(np.median(top)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm), "power_w_max": float(max(pw))}
        return out


# ---------------------------------------------------------------------------
# CPU arm: the reference-shaped oracle loop (24 FFTs / iteration, unfused), REAL iterations at n x n
# ---------------------------------------------------------------------------
def cpu_oracle_steps(n, steps, warmup, workers, model=0, image=None):
    """`warmup` untimed + `steps` timed SAPG main-loop iterations of ONE chain of the oracle at n x n
    (oracle/sapg.py with scipy.fft on `workers` threads and the plain-C TV prox of oracle/c).
    Returns the list of seconds per timed iteration."""
    import scipy.fft
    import oracle
    from oracle import operators as OP
    OP.set_fft(lambda a: scipy.fft.fft2(a, workers=workers), lambda a: scipy.fft.ifft2(a, workers=workers))
    oracle.tv.set_threads(workers)                  # torchrun exports OMP_NUM_THREADS=1
    x = synthetic_truth(n) if image is None else image
    rng = np.random.default_rng(1)
    stamps = []

    def randn(shape):
        stamps.append(time.perf_counter())
        return rng.standard_normal(shape)

    total = steps + warmup
    kw = dict(fix_w1=0, fix_w2=0) if model == 0 else {}
    res = OP.setup_demo(model, x, lambda s: rng.standard_normal(s), samples=total + 1, warmup=1, burnIn=2,
                        evMax=EVMAX, **kw)
    if model == 0:
        oracle.sapg.SAPG_algorithm_Guassian(res[0], res[1], res[2], randn)
    elif model == 1:
        oracle.sapg.SAPG_algorithm_moffat(res[0], res[1], randn)
    else:
        oracle.sapg.SAPG_algorithm_laplace(res[0], res[1], randn)
    stamps.append(time.perf_counter())
    OP.set_fft(np.fft.fft2, np.fft.ifft2)
    return list(np.diff(stamps))[warmup:]


def cpu_sample_text(n, steps, warmup, workers):
    return (f"{steps} timed (+{warmup} untimed) SAPG main-loop iterations of ONE chain of the CPU restatement of the "
            f"reference (oracle/: unfused, 24 FFTs + 25 Chambolle sweeps per iteration) at the full {n}x{n} size, no "
            f"extrapolation; scipy.fft workers={workers}, TV prox = oracle/c (OpenMP, {workers} threads), other "
            f"elementwise work numpy (1 thread); MATLAB/Octave absent so maxNumCompThreads is N/A")


def run_reference(args, rank, world):
    if rank != 0:
        return
    workers = os.cpu_count() or 1
    t0 = time.perf_counter()
    per = cpu_oracle_steps(args.size, args.steps, args.warmup, workers)
    wall = time.perf_counter() - t0
    ms = float(np.mean(per)) * 1e3
    rate = 1e3 / ms                                              # one chain advances one step per iteration
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True,
            "scaling": scaling_kind(args), "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, world),
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": workers, "kind": "port",
                             "sample": cpu_sample_text(args.size, args.steps, args.warmup, workers)},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "step_note": "a reference step = one main-loop iteration of ONE chain (the reference runs one chain); "
                         "chain-steps/s is normalised per chain, so it compares with the GPU arm's value directly",
            "wall_s": wall}
    print(json.dumps(line), flush=True)


def chains_for(args, world):
    if args.chains_per_gpu:
        return args.chains_per_gpu, args.chains_per_gpu * world
    if args.total_chains % world:
        raise SystemExit(f"--total-chains {args.total_chains} is not divisible by {world} ranks")
    return args.total_chains // world, args.total_chains


def scaling_kind(args):
    return "weak" if args.chains_per_gpu else "strong"


def workload_config(args, world):
    nch, tot = chains_for(args, world)
    ws = args.size * args.size * 8 * 9 * nch
    return {"workload": f"synthetic {args.size}x{args.size} Gaussian-PSF SAPG main loop (BASELINE.json configs[3]), "
                        f"{tot} MYULA chains sharded over {world} GPU(s) = {nch} per GPU, Chambolle K={CHAMBOLLE_K}, "
                        f"psf 7x7, BSNR 30, estimating theta/sigma2/w1/w2",
            "image": f"{args.size}x{args.size}", "chains_per_gpu": nch, "total_chains": tot,
            "parallelism": f"chains x{world}",
            "l2_policy": f"working set per step ({ws / 1e9:.1f} GB) far exceeds the 126 MB L2; no flush needed"
            if ws > 4 * 126e6 else "L2 flushed between runs only"}


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def chamb_plan_n4(k=CHAMBOLLE_K):
    """number of 4-level launches in the block plan of sbd.cu chambolle()"""
    a4, r4 = k // 4, k % 4
    if r4 == 1 and a4 >= 2 and os.environ.get("SBD_CHAMB_PLAN33", "1") != "0":
        return a4 - 2
    return a4 if r4 in (1, 3) else a4 - 1


def roofline_block(phases, npix, nch, K, value, world, t_main, sm_mhz=None, seg=128):
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak = 6650.0; peak_src = "fallback 6.65 TB/s (B200_PROFILING.md)"
    n4 = chamb_plan_n4()
    n_prox = int(phases["chambolle_sweeps"][1])
    launches_timed = n_prox * n4
    sweep_ms = phases["chambolle_sweeps"][0] * n_prox / K / max(launches_timed, 1)      # phases[..][0] is scaled to K steps
    sweep_bytes = 40.0 * npix * nch * 4                        # algorithmic bytes of the 4 sweeps one launch applies
    achieved = sweep_bytes / (sweep_ms * 1e-3) / 1e9 if sweep_ms > 0 else 0.0
    # measured DRAM traffic per launch: ncu --set full captures, per pixel and chain (profiles/roofline_traffic.json)
    prof = {}
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        try:
            prof = json.load(open(tp))
        except Exception:
            prof = {}
    traffic = None
    key = f"k_chamb_multi4:{int(round(npix ** 0.5))}x{nch}"
    if key in prof.get("per_launch_bytes", {}):
        traffic = float(prof["per_launch_bytes"][key])
    dram_frac = (traffic / (sweep_ms * 1e-3) / 1e9 / peak) if (traffic and sweep_ms > 0) else None
    issue = prof.get("issue_model", {})
    issue_frac = None
    if issue and sweep_ms > 0:
        # cycles the SMSP issue ports need for one launch (tools/fp64_microbench.cu calibration) / measured cycles
        trips = npix * nch / (2.0 * 56.0)                        # warp-trips: 2 rows x 56 output pixels x 4 levels each
        # instructions outside the steady-state loop: measured 1.151x at 128-row segments (ncu); the part that is the
        # vertical halo of a segment shrinks with the segment length the run uses
        overhead = 1.03 + (issue.get("overhead", 1.151) - 1.03) * 128.0 / max(seg, 128)
        cyc_needed = trips * (issue["fp64_per_trip"] * issue["fp64_issue_cycles"] + issue["other_per_trip"]) \
            * overhead / (148 * 4)
        clk = (sm_mhz or issue.get("sm_clock_mhz", 1920.0)) * 1e6
        issue_frac = cyc_needed / (sweep_ms * 1e-3 * clk)
    step_alg_gbs = alg_bytes_per_chain_step(npix) * value / 1e9 / world
    step_traffic = prof.get("step_bytes_per_pixel_chain")
    step_dram_gbs = (step_traffic * npix * nch * K / t_main / 1e9) if step_traffic else None
    return {
        "bound": "hbm", "bound_measured": "fp64_issue",
        "kernel": "k_chamb_multi<4> (4 Chambolle sweeps fused per launch)",
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_model": achieved / peak,
        "traffic": traffic, "dram_frac": dram_frac, "issue_frac": issue_frac,
        "peak_source": peak_src, "bytes_per_launch": sweep_bytes, "ms_per_launch": sweep_ms,
        "launches_timed": launches_timed,
        "step": {"alg_gbs_per_gpu": step_alg_gbs, "alg_frac_of_hbm_peak": step_alg_gbs / peak,
                 "dram_gbs_per_gpu": step_dram_gbs,
                 "dram_frac_of_hbm_peak": (step_dram_gbs / peak) if step_dram_gbs else None},
        "note": "achieved/frac use the ALGORITHMIC bytes of SURVEY.md 8(d) (40 B/pixel/sweep x the 4 sweeps of one launch). "
                "The launch keeps its 4 sweep levels in registers (temporal blocking), so its measured DRAM traffic "
                "(`traffic`, ncu) is ~1/4 of that and `frac` exceeds 1: the kernel is NOT HBM-bound. `dram_frac` = measured "
                "traffic / live time / peak is its real DRAM utilisation; what bounds it is fp64 instruction issue "
                "(`issue_frac` = issue-port cycles needed by the SASS instruction mix of profiles/*chamb*sass*, calibrated "
                "with tools/fp64_microbench.cu, over measured cycles). `step` gives the same two readings for the whole MYULA step."}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import sbd_b200
    from sbd_b200 import host as H
    from sbd_b200._lib import lib, sbd_traces, c_double_p

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n = args.size
    nch, total = chains_for(args, world)
    npix = n * n
    K, W = args.steps, args.warmup
    shard = sbd_b200.ChainShard(total, world, rank)

    # ---- synthetic problem (same on every rank)
    x_true = synthetic_truth(n)
    eng = sbd_b200.Engine(n, n, 7, H.GAUSSIAN, 0.0, nch, local_rank)
    shard.init_engine_comm(eng)
    Ax = eng.blur(x_true, PSI_TRUE, H.OP_A)
    nrm = float(np.linalg.norm(Ax - Ax.mean()))
    sig = lambda b: nrm / np.sqrt(npix * 10 ** (b / 10))    # run_Gaussian_demo.m:148-152
    sigma, smin, smax = sig(30), sig(15), sig(45)
    y = Ax + sigma * np.random.default_rng(2).standard_normal((n, n))
    del Ax

    def params(samples, warmup):
        op, c = gaussian_op(n, sigma, smin, smax, EVMAX, samples, warmup)
        return H.make_params(H.GAUSSIAN, op, c, n_chains=nch, seed=1, chain_offset=shard.chain_offset,
                             total_chains=shard.total_chains)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- (1) value: y resident in HBM, device-timed main loop
    y_dev = torch.from_numpy(np.ascontiguousarray(y.T)).cuda()      # column-major image on the device
    prm = params(K + 1, W + 1)
    tr = sbd_traces()
    th = np.zeros(K + 1); tr.thetas = th.ctypes.data_as(c_double_p)
    s2 = np.zeros(K + 1); tr.sigmas = s2.ctypes.data_as(c_double_p)
    ck = np.zeros(K + 1, dtype=np.int32); tr.chambolle_iters = ck.ctypes.data_as(C.POINTER(C.c_int32))
    dump = {f: np.zeros(K + 1) for f in DUMP_TRACES} if args.dump_outputs else {}
    for f, b in dump.items():                                 # copied back after the clock stops
        setattr(tr, f, b.ctypes.data_as(c_double_p))
    barrier()
    clocks = ClockSampler(local_rank) if rank == 0 else None
    rc = lib.sbd_sapg_run_dev(eng._h, y_dev.data_ptr(), None, C.byref(prm), C.byref(tr))
    if rc != 0:
        raise RuntimeError(lib.sbd_last_error(eng._h).decode())
    barrier()
    clk = clocks.stop() if clocks else None
    t_main = max_over_ranks(tr.seconds_main)
    launches = int(tr.launches_main)
    if args.dump_outputs:
        # The timed run leaves the chains' last samples on the device.  The same run (same inputs, seed and summation
        # order, so bit-identical) is repeated untimed with their copy-out switched on, and must reproduce the timed
        # trajectories.
        xl = torch.empty(nch * npix, dtype=torch.float64).pin_memory()
        tr_x = sbd_traces()
        th_x = np.zeros(K + 1); tr_x.thetas = th_x.ctypes.data_as(c_double_p)
        s2_x = np.zeros(K + 1); tr_x.sigmas = s2_x.ctypes.data_as(c_double_p)
        tr_x.X_last = C.cast(xl.data_ptr(), c_double_p)
        rc = lib.sbd_sapg_run_dev(eng._h, y_dev.data_ptr(), None, C.byref(prm), C.byref(tr_x))
        if rc != 0:
            raise RuntimeError(lib.sbd_last_error(eng._h).decode())
        if not (np.array_equal(th_x, th) and np.array_equal(s2_x, s2)):
            raise RuntimeError("--dump-outputs: the repeated main loop did not reproduce the timed one")
        idx = last_sample_pixels(npix, nch)
        dump.update(thetas=th, sigmas=s2, chambolle_iters=ck, X_last_sample_index=idx,
                    X_last_sample=xl.numpy().reshape(nch, npix)[:, idx])
        del xl
    # per-phase CUDA-event times come from a second, short run with the phase timers on: profiling serialises the
    # two streams of an iteration (prox next to analysis + gradient), so it is kept out of the headline number
    KP = min(K, 4)
    prm_p = params(KP + 1, 2)
    tr_p = sbd_traces()
    eng.set_profile(True)
    rc = lib.sbd_sapg_run_dev(eng._h, y_dev.data_ptr(), None, C.byref(prm_p), C.byref(tr_p))
    if rc != 0:
        raise RuntimeError(lib.sbd_last_error(eng._h).decode())
    barrier()
    phases = {k_: (v_[0] * K / KP, v_[1]) for k_, v_ in eng.phase_times().items()}     # scaled to K steps
    t_serial = max_over_ranks(tr_p.seconds_main) / KP
    eng.set_profile(False)
    value = K * shard.total_chains / t_main
    eng.set_option("geom_chains", shard.total_chains)
    chamb_seg = eng.geometry(nch)["chamb_seg"]               # segment length the run used (derived from the total)
    eng.set_option("geom_chains", 0)
    sweeps_executed = int(ck[1:].sum())                      # chain 0's stop behaviour (all chains share theta)

    # ---- (2) e2e: host-pointer C ABI, pinned host buffers, copies inside the timed region
    y_pin = torch.from_numpy(np.ascontiguousarray(y.T)).pin_memory()
    xl_pin = torch.empty(nch * npix, dtype=torch.float64).pin_memory()
    prm2 = params(K + 1, 1)
    tr2 = sbd_traces()
    bufs = {k: np.zeros(K + 1) for k in ("thetas", "sigmas", "psi0", "psi1", "logPiTraceX", "gXTrace")}
    for k_, b in bufs.items():
        setattr(tr2, k_, b.ctypes.data_as(c_double_p))
    tr2.X_last = C.cast(xl_pin.data_ptr(), c_double_p)
    barrier()
    t0 = time.perf_counter()
    rc = lib.sbd_sapg_run(eng._h, C.cast(y_pin.data_ptr(), c_double_p), None, None, C.byref(prm2), None, C.byref(tr2))
    if rc != 0:
        raise RuntimeError(lib.sbd_last_error(eng._h).decode())
    torch.cuda.synchronize()
    wall = max_over_ranks(time.perf_counter() - t0)
    e2e_value = K * shard.total_chains / wall
    h2d = npix * 8 / K
    d2h = (nch * npix * 8 + 6 * (K + 1) * 8) / K
    e2e_main_s = tr2.seconds_main
    del xl_pin, y_pin, y_dev
    eng.close()

    # ---- configs[2] (N > 1): Laplace SAPG, one images/*.png per GPU, replicas, no collective
    cfg2 = None
    if world > 1 and not args.no_extras:
        cfg2 = config2_laplace(rank, world, local_rank, barrier, max_over_ranks)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": t_main / K * 1e3,
        "higher_is_better": True, "scaling": scaling_kind(args), "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "wall_s": wall, "device_main_loop_s": e2e_main_s,
                "note": "one sbd_sapg_run call = K steps; y from pinned host memory in, trajectories + every chain's last "
                        "sample out (pinned), wall clock around the call, max over ranks"},
        "gpu_launches": launches,
        "clocks": clk,
        "roofline": roofline_block(phases, npix, nch, K, value, world, t_main, (clk or {}).get("sm_mhz"), chamb_seg),
        "fused_step": {"alg_bytes_per_chain_step": alg_bytes_per_chain_step(npix),
                       "phase_ms_per_step": {("chambolle_total" if k_ == "chambolle_other" else k_): v_[0] / K
                                             for k_, v_ in phases.items()},
                       "ms_per_step_serial_order": t_serial * 1e3,
                       "note": "phase times from a separate profiled run in serial order; in the headline run the prox of "
                               "an iteration runs on its own stream next to the analysis / scalar update / next gradient"},
        "sweeps_executed_chain0": sweeps_executed,
        "theta_last": float(th[-1]), "sigma2_last": float(s2[-1]),
    }
    if cfg2:
        line["config2_laplace_one_image_per_gpu"] = cfg2
    if world == 1 and not args.no_size_sweep:
        # the metric is quoted on 256^2 .. 4096^2: short runs of the same SAPG main loop at the smaller sizes (8 chains)
        sweep = {}
        for m in (2048, 1024, 512, 256):
            if m >= n:
                continue
            sweep[str(m)] = round(quick_rate(m, 8, local_rank), 2)
        line["size_sweep_chain_steps_per_s_8chains"] = sweep
    if world == 1 and not args.no_extras:
        try:
            line["config0_cman256_full_demo"] = config0_cman(local_rank, args)
            line["config1_moffat_boat512"] = config1_moffat(local_rank)
            line["config4_operator_sweep"] = config4_operators(local_rank)
        except Exception as e:                                   # extras must never take the headline line down
            line["extras_error"] = repr(e)
    if world == 1 and not args.no_cpu_baseline:
        workers = os.cpu_count() or 1
        cs, cw = 3, 1
        per = cpu_oracle_steps(n, cs, cw, workers)
        rate = 1.0 / float(np.mean(per))
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": workers, "kind": "port",
                                "s_per_iteration": [round(float(p), 3) for p in per],
                                "sample": cpu_sample_text(n, cs, cw, workers)}
    if args.dump_outputs:
        write_dump(args.dump_outputs, dump)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def quick_rate(n, nch, device, steps=30, warmup=4):
    """chain-steps/s of the SAPG main loop at n x n (device-resident y, CUDA-graph replay), same model as the headline."""
    import torch
    import sbd_b200
    from sbd_b200 import host as H
    from sbd_b200._lib import lib, sbd_traces
    eng = sbd_b200.Engine(n, n, 7, H.GAUSSIAN, 0.0, nch, device)
    x = synthetic_truth(n)
    Ax = eng.blur(x, PSI_TRUE, H.OP_A)
    nrm = float(np.linalg.norm(Ax - Ax.mean()))
    sig = lambda b: nrm / np.sqrt(n * n * 10 ** (b / 10))
    y = Ax + sig(30) * np.random.default_rng(2).standard_normal((n, n))
    op, c = gaussian_op(n, sig(30), sig(15), sig(45), EVMAX, steps + 1, warmup + 1)
    op["use_graph"] = 1
    prm = H.make_params(H.GAUSSIAN, op, c, n_chains=nch, seed=1)
    y_dev = torch.from_numpy(np.ascontiguousarray(y.T)).cuda()
    tr = sbd_traces()
    rc = lib.sbd_sapg_run_dev(eng._h, y_dev.data_ptr(), None, C.byref(prm), C.byref(tr))
    if rc != 0:
        raise RuntimeError(lib.sbd_last_error(eng._h).decode())
    rate = steps * nch / tr.seconds_main
    eng.close()
    return rate


# ---------------------------------------------------------------------------
# the other BASELINE.json configs (extra keys of the same JSON line)
# ---------------------------------------------------------------------------
def psnr(x, z):
    return float(10 * np.log10(255.0 ** 2 / np.mean((x - z) ** 2)))


def config0_cman(device, args):
    """configs[0]: run_Gaussian_demo.m on cameraman 256x256 with the reference's run lengths (warm-up 15000 +
    20000 SAPG iterations = 34 998 MYULA steps, run_Gaussian_demo.m:47,50), theta / sigma^2 / w1 / w2 estimated,
    one chain, CUDA-graph replay; the CPU leg times REAL 256x256 iterations of the oracle on this host."""
    from sbd_b200 import demo, host as H
    x = np.load(golden("cman_u8.npy")).astype(np.float64)
    t0 = time.perf_counter()
    res = demo.run_demo(H.GAUSSIAN, x, map_estimate=True, post_mean=True, use_graph=True, fix_w1=0, fix_w2=0,
                        seed=1, device=device, samples=args.cman_samples, warmup=args.cman_warmup, name="cman")
    wall = time.perf_counter() - t0
    steps = (args.cman_warmup - 1) + (args.cman_samples - 1)
    workers = os.cpu_count() or 1
    per = cpu_oracle_steps(256, 40, 3, workers, image=x)
    cpu_s = float(np.mean(per))
    return {"config": "run_Gaussian_demo.m on cman 256x256, fix_w1 = fix_w2 = 0, 1 chain, use_graph",
            "myula_steps": steps, "gpu_sapg_device_s": res["execTimeFindParameters"], "gpu_sapg_wall_s": res["SAPG_time"],
            "gpu_total_wall_s_with_setup_and_MAP": wall, "gpu_steps_per_s": steps / res["execTimeFindParameters"],
            "theta_EB": res["theta_EB"], "w1_EB": res["w1_EB"], "w2_EB": res["w2_EB"], "sigma2_EB": res["sigma_EB"],
            "true": {"w1": 0.4, "w2": 0.3, "sigma2": res["sigma"] ** 2},
            "psnr_y": psnr(x, res["y"]), "psnr_mmse": psnr(x, res["posteriormean"]), "psnr_map": psnr(x, res["xMAP"]),
            "cpu_s_per_step_measured_256": cpu_s, "cpu_cores": workers, "cpu_steps_timed": len(per),
            "cpu_s_for_the_same_steps": cpu_s * steps, "speedup_vs_cpu": cpu_s * steps / res["execTimeFindParameters"],
            "target": ">= 100x (BASELINE.json north_star)"}


def config1_moffat(device, samples=1500, warmup=500):
    """configs[1]: run_moffat_demo.m on boat 512x512, (alpha, beta) semi-blind, single GPU, one chain."""
    from sbd_b200 import demo, host as H
    x = np.load(golden("boat_u8.npy")).astype(np.float64)
    res = demo.run_demo(H.MOFFAT, x, map_estimate=False, use_graph=True, seed=1, device=device, samples=samples,
                        warmup=warmup, name="boat")
    steps = (warmup - 1) + (samples - 1)
    workers = os.cpu_count() or 1
    per = cpu_oracle_steps(512, 6, 2, workers, model=1, image=x)
    cpu_s = float(np.mean(per))
    return {"config": f"run_moffat_demo.m on boat 512x512, warm-up {warmup} + {samples} SAPG iterations, 1 chain, use_graph",
            "myula_steps": steps, "gpu_device_s": res["execTimeFindTheta"], "gpu_steps_per_s": steps / res["execTimeFindTheta"],
            "alpha_last": float(res["alphas"][-1]), "beta_last": float(res["betas"][-1]), "true": {"alpha": 0.4, "beta": 3.5},
            "cpu_s_per_step_measured_512": cpu_s, "cpu_cores": workers,
            "speedup_vs_cpu": cpu_s * steps / res["execTimeFindTheta"]}


def config4_operators(device, sizes=(256, 512, 1024, 2048, 4096), batch=256):
    """configs[4]: fused FFT blur A / A' and the 20-iteration Chambolle prox on a batch of 256 images, device resident,
    CUDA events (the batch is processed in sub-batches that fit HBM)."""
    import torch
    import sbd_b200
    from sbd_b200 import host as H
    from sbd_b200._lib import lib
    out = {}
    psi = (C.c_double * 2)(0.4, 3.5)
    for n in sizes:
        npix = n * n
        sub = max(1, min(batch, int(24e9 // (npix * 8 * 11))))
        eng = sbd_b200.Engine(n, n, 7, H.MOFFAT, 0.0, sub, device)
        x = torch.rand(sub, n, n, dtype=torch.float64, device="cuda") * 255.0
        o = torch.empty_like(x)
        nsub = (batch + sub - 1) // sub

        def timed(fn):
            fn(); lib.sbd_synchronize(eng._h); torch.cuda.synchronize()
            best = 1e30
            for _ in range(2):
                t0 = time.perf_counter()
                for _ in range(nsub):
                    fn()
                lib.sbd_synchronize(eng._h)
                best = min(best, time.perf_counter() - t0)
            return best

        def chk(rc):
            if rc != 0:
                raise RuntimeError(lib.sbd_last_error(eng._h).decode())

        tA = timed(lambda: chk(lib.sbd_blur_dev(eng._h, x.data_ptr(), psi, 0, o.data_ptr(), sub)))
        tAT = timed(lambda: chk(lib.sbd_blur_dev(eng._h, x.data_ptr(), psi, 1, o.data_ptr(), sub)))
        tP = timed(lambda: chk(lib.sbd_tvprox_dev(eng._h, x.data_ptr(), 0.5, 20, 0.0, 0.249, o.data_ptr(), None, None, sub)))
        nimg = nsub * sub
        out[str(n)] = {"sub_batch": sub, "A_images_per_s": nimg / tA, "AT_images_per_s": nimg / tAT,
                       "prox20_images_per_s": nimg / tP,
                       "A_alg_gbs": 64.0 * npix * nimg / tA / 1e9, "prox20_alg_gbs": 832.0 * npix * nimg / tP / 1e9}
        eng.close()
        del x, o
    out["note"] = ("host wall clock around nsub back-to-back device-resident calls + one stream sync; algorithmic bytes: "
                   "A or A' = 64 B/pixel (two real<->half-spectrum round trips), Chambolle-20 prox = 832 B/pixel (per-sweep model)")
    return out


def config2_laplace(rank, world, local_rank, barrier, max_over_ranks, samples=400, warmup=200):
    """configs[2]: run_laplace_demo.m over the 8 images/*.png, one image per GPU (rank r takes image r mod 8),
    replicas only - no data-path collective."""
    from sbd_b200 import demo, host as H
    imgs = np.load(golden("images_u8.npz"))
    names = sorted(imgs.files)
    name = names[rank % len(names)]
    x = imgs[name].astype(np.float64)
    eng = H.Engine(x.shape[0], x.shape[1], 7, H.LAPLACE, 0.0, 1, local_rank)
    barrier()
    t0 = time.perf_counter()
    res = demo.run_demo(H.LAPLACE, x, engine=eng, map_estimate=False, use_graph=True, seed=1 + rank, samples=samples,
                        warmup=warmup, name=name)
    dev_s = max_over_ranks(res["execTimeFindTheta"])
    wall = max_over_ranks(time.perf_counter() - t0)
    eng.close()
    steps = (warmup - 1) + (samples - 1)
    return {"config": f"run_laplace_demo.m, one 512x512 images/*.png per GPU ({world} GPUs, replicas, no collective), "
                      f"warm-up {warmup} + {samples} SAPG iterations each",
            "image_steps_per_s_device": world * steps / dev_s, "image_steps_per_s_wall_with_setup": world * steps / wall,
            "rank0_image": names[0], "rank0_b_last": float(res["bs"][-1]), "true_b": 0.3,
            "rank0_mean_chambolle_sweeps": float(np.mean(res["chambolle_iters"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--total-chains", type=int, default=64, help="chains over all GPUs (strong scaling, configs[3])")
    ap.add_argument("--chains-per-gpu", type=int, default=0, help="> 0: weak scaling with this many chains on every GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-size-sweep", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[0]/[1]/[2]/[4] extra keys")
    ap.add_argument("--cman-samples", type=int, default=20000)
    ap.add_argument("--cman-warmup", type=int, default=15000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed main loop's trajectories and a seeded sample of its chains' last samples "
                         "as DIR/<name>.npy (float64; the sample and its indices take 32 MiB at most)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
