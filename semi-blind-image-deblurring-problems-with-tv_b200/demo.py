"""Host-side mirror of the reference's experiment scripts, on top of the CUDA engine.

  run_Gaussian_demo.m:34-260   cameraman / images/*.png, Gaussian PSF (w1, w2)
  run_moffat_demo.m:34-240     Moffat PSF (alpha, beta)
  run_laplace_demo.m:34-205    Laplace PSF (b)

Every numerical step runs on the GPU through the C ABI (include/sbd.h): the power
iteration for evMax (`sbd_max_eigenval`), the observation synthesis (`sbd_observe`),
SAPG (`sbd_sapg_run`) and the post-SAPG MAP estimate (`sbd_salsa_tv`).  What is
left on the host is what the scripts do in scalar MATLAB: option structs, step
sizes, the `for snr` / `for i_im` loops and saving the results
(`run_batch`, SURVEY.md 8 f4; legacy `save` at SALSA/run_deblur_tv.m:166).
There is no CPU fallback: without libsbd.so and a B200 every call raises.
"""
import os
import time

import numpy as np

from . import host as H

# run_Gaussian_demo.m:34-85 / run_moffat_demo.m:34-83 / run_laplace_demo.m:34-70
DEFAULTS = {
    H.GAUSSIAN: dict(samples=20000, warmup=15000, lambdaMax=2.0, gammaFrac=0.98,
                     min_th=1e-3, max_th=1.0, min_w1=0.1, max_w1=1.0, min_w2=0.1, max_w2=1.0,
                     BSNR_max=45, BSNR_min=15, BSNR=30, th_init=0.01, w1_init=0.5, w2_init=0.3,
                     d_exp=0.8, psf_size=7, phi=0.0, w1=0.4, w2=0.3, fix_w1=1, fix_w2=1, fix_sigma=0),
    H.MOFFAT: dict(samples=20000, warmup=15000, lambdaMax=2.0, gammaFrac=0.98,
                   min_th=1e-3, max_th=1.0, min_alpha=1e-2, max_alpha=1.0, min_beta=0.1, max_beta=10.0,
                   BSNR_max=35, BSNR_min=18, BSNR=30, psf_size=7, th_init=0.01, alpha_init=1.0,
                   beta_init=10.0, d_exp=0.8, alpha=0.4, beta=3.5, fix_alpha=0, fix_beta=0, fix_sigma=0),
    H.LAPLACE: dict(samples=20000, warmup=15000, lambdaMax=0.1, gammaFrac=0.98,
                    min_th=1e-3, max_th=1.0, th_init=0.01, min_b=1e-3, max_b=1.0, b_init=0.1,
                    BSNR_max=45, BSNR_min=15, BSNR=30, psf_size=7, d_exp=0.8, b=0.3, fix_b=0, fix_sigma=0),
}
C_GAUSSIAN = dict(sigma=1000.0, theta=0.01, w1=10.0, w2=10.0, lam=1.0, gam=1.0)      # run_Gaussian_demo.m:34-39
_NAMES = {H.GAUSSIAN: ("w1", "w2"), H.MOFFAT: ("alpha", "beta"), H.LAPLACE: ("b",)}
_EV_PARAMS = {H.GAUSSIAN: (1.0, 1.0), H.MOFFAT: (1.0, 5.0), H.LAPLACE: (1.0,)}      # demo :142 / :140 / :110
MODEL_NAMES = {H.GAUSSIAN: "gaussian", H.MOFFAT: "moffat", H.LAPLACE: "laplace"}


def setup_demo(model, x, engine=None, noise=None, x0_eig=None, seed=1, chambolleit=25, evMax=None, device=0,
               **overrides):
    """Everything the demo script does between `imread` and the SAPG call, on the device:
    evMax by power iteration (utils/max_eigenval_*.m), Ax, sigma from the BSNR, y = Ax + sigma*noise
    (run_Gaussian_demo.m:142-168), then Lf / lambda / gamma (:177-184).
    `noise` / `x0_eig` (rows x cols) replace MATLAB's randn stream; None -> on-device Philox(seed).
    Returns (y, op, engine) with `op` the plain-data part of the reference's struct."""
    x = np.asarray(x, dtype=np.float64)
    op = dict(DEFAULTS[model])
    op.update(overrides)
    op.setdefault("burnIn", (op["samples"] * 80) // 100)                 # :49
    op.setdefault("d_scale", 0.01 / op["th_init"])                       # :72
    names = _NAMES[model]
    for n in names:
        if op["fix_" + n]:
            op[n + "_init"] = op[n]                                      # :102-107
    eng = engine or H.engine_for(x.shape, op["psf_size"], model, op.get("phi", 0.0), device=device)
    if evMax is None:
        evMax, _ = eng.max_eigenval(_EV_PARAMS[model], 1e-4, 10000, x0=x0_eig, seed=seed)   # :142
    op["evMax"] = float(evMax)
    true_psi = tuple(op[n] for n in names)
    y, sigma, nrm = eng.observe(x, true_psi, op["BSNR"], noise=noise, seed=seed)             # :145-168
    dimX = x.size
    sig = lambda b: nrm / np.sqrt(dimX * 10 ** (b / 10))                                     # :148-152
    sigma_min, sigma_max = sig(op["BSNR_min"]), sig(op["BSNR_max"])
    op["sigma"] = sigma
    op["sigma_init"] = sigma ** 2 if op["fix_sigma"] else (sigma_min ** 2 + sigma_max ** 2) / 2   # :157-161
    op["sigma_min"], op["sigma_max"] = sigma_min ** 2, sigma_max ** 2                        # :162-163
    Lf = lambda s2: op["evMax"] ** 2 / s2                                                    # :178
    if model == H.LAPLACE:
        op["Lf"] = max(Lf(op["sigma_min"]), Lf(op["sigma_max"]))         # run_laplace_demo.m:137
    else:
        op["Lf"] = min(Lf(op["sigma_min"]), Lf(op["sigma_max"]))         # run_Gaussian_demo.m:179
    op["lambda"] = min(5 / op["Lf"], op["lambdaMax"])                    # :182
    op["gamma_max"] = 1 / (op["Lf"] + 1 / op["lambda"])                  # :183
    op["gamma"] = (10 if model == H.LAPLACE else 1) * op["gammaFrac"] * op["gamma_max"]      # :184 / laplace :142
    op["chambolleit"] = chambolleit                                      # :188
    op["x"] = x
    if model == H.LAPLACE:
        op["X0"] = y                                                     # run_laplace_demo.m:127
    return y, op, eng


def run_demo(model, x, engine=None, map_estimate=True, n_chains=1, seed=1, noise_sapg=None, post_mean=False,
             use_graph=True, name="", post_levels=0, post_batch=0, post_ci=0.0, **kw):
    """One pass of the body of the experiment loops (run_Gaussian_demo.m:100-242): observation, SAPG,
    SALSA MAP estimate with the empirical-Bayes parameters, MSE.  Returns the `results` dict the script
    saves, plus timings.  post_levels > 0 adds the posterior statistics (host.Engine.sapg), post_batch (-1 or a batch
    length, with post_levels) their ESS, MCSE and split-Rhat, post_ci = alpha (with post_levels) the median and the
    (1 - alpha) credible interval."""
    t0 = time.perf_counter()
    y, op, eng = setup_demo(model, x, engine=engine, seed=seed, **kw)
    if n_chains > eng.max_batch:
        raise ValueError("n_chains exceeds the engine's max_batch")
    op["use_graph"] = int(bool(use_graph))
    t1 = time.perf_counter()
    names = _NAMES[model]
    if model == H.GAUSSIAN:
        th, p0, p1, s2, r = H.SAPG_algorithm_Guassian(y, op, dict(C_GAUSSIAN), noise=noise_sapg, n_chains=n_chains,
                                                      seed=seed, engine=eng, post_mean=post_mean,
                                                      post_levels=post_levels, post_batch=post_batch, post_ci=post_ci)
        psi_eb = (p0, p1)
    elif model == H.MOFFAT:
        th, p0, p1, s2, r = H.SAPG_algorithm_moffat(y, op, noise=noise_sapg, n_chains=n_chains, seed=seed, engine=eng,
                                                    post_mean=post_mean, post_levels=post_levels,
                                                    post_batch=post_batch, post_ci=post_ci)
        psi_eb = (p0, p1)
    else:
        th, p0, s2, r = H.SAPG_algorithm_laplace(y, op, noise=noise_sapg, n_chains=n_chains, seed=seed, engine=eng,
                                                 post_mean=post_mean, post_levels=post_levels,
                                                 post_batch=post_batch, post_ci=post_ci)
        psi_eb = (p0,)
    t2 = time.perf_counter()
    res = dict(r)
    res.update(name=name, model=MODEL_NAMES[model], x=x, y=y, theta_EB=th, sigma_EB=s2, sigma=op["sigma"],
               SAPG_time=t2 - t1, setup_time=t1 - t0, evMax=op["evMax"])
    for n, v in zip(names, psi_eb):
        res[n + "_EB"] = v
        res[n] = op[n]
    if map_estimate:
        mu = th / 10                                                     # :220
        sal = eng.salsa_tv(y, psi_eb, th * s2, mu, maxiter=500, tolA=1e-5, tv_iters=10, x_true=x)    # :229-242
        xmap = sal["x"]
        res["xMAP"] = xmap
        res["mse"] = 10 * np.log10(np.linalg.norm(x - xmap, "fro") ** 2 / x.size)                    # :244
        res["salsa_outer"] = sal["n_outer"]
        res["MAP_time"] = time.perf_counter() - t2
    return res


def _savable(res):
    out = {}
    for k, v in res.items():
        if isinstance(v, (int, float, str, np.ndarray, np.floating, np.integer)):
            out[k] = v
        elif k == "options":
            for kk, vv in v.items():
                if isinstance(vv, (int, float, str, np.floating, np.integer)):
                    out["op_" + kk] = vv
        elif k == "posterior":                  # one entry per block size s
            for p in v:
                out[f"posterior_std_s{p['scale']}"] = p["std"]
                out[f"Rhat_s{p['scale']}"] = p["Rhat"]
                if "ESS" in p:                  # post_batch
                    for q in ("ESS", "MCSE", "Rhat_split"):
                        out[f"{q}_s{p['scale']}"] = p[q]
                if "ci_width" in p:             # post_ci
                    out[f"CI_width_s{p['scale']}"] = p["ci_width"]
    return out


def run_batch(model, images, bsnrs=(30,), out_dir=None, rank=0, world=1, device=None, **kw):
    """The experiment loops `for snr = [...]` / `for i_im = [...]` (run_Gaussian_demo.m:98-100,
    run_moffat_demo.m:105-107, run_laplace_demo.m:73-80) as a batch driver.  `images` maps a name to a
    2-D array.  Jobs (snr, image) are dealt round-robin to `world` ranks - one process per GPU, replicas
    only, no collective (BASELINE.json configs[2]: one image per GPU) - and each result is saved to
    `out_dir/<model>_<name>_bsnr<snr>.npz` (the scripts' `save`).  Returns {(name, snr): results} of this rank."""
    jobs = [(snr, name) for snr in bsnrs for name in images]
    mine = jobs[rank::world]
    dev = rank if device is None else device
    out = {}
    engines = {}
    for snr, name in mine:
        x = np.asarray(images[name], dtype=np.float64)
        key = x.shape
        if key not in engines:
            opts = dict(DEFAULTS[model]); opts.update(kw)
            engines[key] = H.Engine(x.shape[0], x.shape[1], opts["psf_size"], model, opts.get("phi", 0.0),
                                    max_batch=kw.get("n_chains", 1), device=dev)
        res = run_demo(model, x, engine=engines[key], name=name, BSNR=snr, **kw)
        out[(name, snr)] = res
        if out_dir:
            os.makedirs(out_dir, exist_ok=True)
            np.savez(os.path.join(out_dir, f"{MODEL_NAMES[model]}_{name}_bsnr{snr}.npz"), **_savable(res))
    for e in engines.values():
        e.close()
    return out
