"""GPU tests of the posterior statistics (include/sbd.h sbd_set_posterior / sbd_posterior_stats, DESIGN.md "Posterior
statistics"): exact against oracle/posterior.py on the device's own samples, existing outputs untouched, graph /
eager / serial streams bitwise identical, against the oracle SAPG, a large shape, the error paths, 2-GPU merge and
the MEX gateway."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import rel, ROOT

pytestmark = pytest.mark.gpu

TOL = 1e-12
TRAJ_TOL = 1e-6
KEYS = ("mean", "within", "between", "var", "std")
TRAJ = ("thetas", "sigmas", "psi0", "psi1", "grad_theta", "grad_psi0", "grad_psi1", "grad_sigma", "logPiTraceX",
        "gXTrace", "err_psf", "tol_theta", "tol_psi0", "tol_psi1", "tol_sigma", "mean_theta", "mean_psi0", "mean_psi1",
        "mean_sigma", "chambolle_iters", "EB")


@pytest.fixture(scope="module")
def sbd():
    import sbd_b200
    return sbd_b200


def _crop(img, shape):
    reps = (-(-shape[0] // img.shape[0]) + 1, -(-shape[1] // img.shape[1]) + 1)
    t = np.block([[img if (i + j) % 2 == 0 else img[::-1, ::-1] for j in range(reps[1])] for i in range(reps[0])])
    return np.ascontiguousarray(t[:shape[0], :shape[1]])


def _problem(sbd, eng, x, burnIn, samples, warmup=3, n_chains=1, seed=7):
    """Moffat SAPG problem built on the device: y = A x + noise, the demo's step sizes; Philox noise for the chains."""
    from sbd_b200 import host as H
    rows, cols = x.shape
    Ax = eng.blur(x, (0.4, 3.5), H.OP_A)
    nrm = float(np.linalg.norm(Ax - Ax.mean()))
    sig = lambda b: nrm / np.sqrt(rows * cols * 10 ** (b / 10))
    y = Ax + sig(30) * np.random.default_rng(2).standard_normal((rows, cols))
    op = dict(samples=samples, warmup=warmup, burnIn=burnIn, psf_size=7, min_th=1e-3, max_th=1.0, th_init=0.01,
              alpha_init=1.0, beta_init=10.0, min_alpha=1e-2, max_alpha=1.0, min_beta=0.1, max_beta=10.0,
              alpha=0.4, beta=3.5, fix_alpha=0, fix_beta=0, fix_sigma=0, d_exp=0.8, d_scale=1.0,
              sigma=sig(30), sigma_init=(sig(18) ** 2 + sig(35) ** 2) / 2, sigma_min=sig(18) ** 2, sigma_max=sig(35) ** 2)
    Lf = min(0.993 ** 2 / op["sigma_min"], 0.993 ** 2 / op["sigma_max"])
    op["lambda"] = min(5 / Lf, 2.0)
    op["gamma"] = 0.98 / (Lf + 1 / op["lambda"])
    return y, lambda post_mean=False, **kw: H.make_params(H.MOFFAT, dict(op, **kw), None, n_chains=n_chains, seed=seed,
                                                          post_mean=post_mean)


def _exact(sbd, x, n_chains, levels, burnIn=2, extra=6):
    """Runs with samples = burnIn+1 .. burnIn+extra return the exact device samples X_ii as their last samples;
    the statistics of the longest run are compared with oracle/posterior.py on them."""
    from oracle import posterior as OP
    eng = sbd.Engine(x.shape[0], x.shape[1], 7, sbd.MOFFAT, 0.0, max_batch=n_chains)
    y, mk = _problem(sbd, eng, x, burnIn, burnIn + extra, n_chains=n_chains)
    runs = [eng.sapg(y, mk(samples=burnIn + k), want_X_warm=False, post_levels=levels if k == extra else 0)
            for k in range(1, extra + 1)]
    longest = runs[-1]
    for r in runs[:-1]:
        S = len(r["thetas"])
        assert np.array_equal(r["thetas"], longest["thetas"][:S])        # the shorter runs are prefixes
        assert np.array_equal(r["sigmas"], longest["sigmas"][:S])
    samples = np.stack([r["X_last"] for r in runs])                       # [extra, C, rows, cols]
    want = OP.stats(samples, levels)
    got = longest["posterior"]
    assert len(got) == levels
    for j, (g, w) in enumerate(zip(got, want)):
        assert g["scale"] == 1 << j and g["n"] == extra and g["chains"] == n_chains
        assert g["mean"].shape == w["mean"].shape == (-(-x.shape[0] // (1 << j)), -(-x.shape[1] // (1 << j)))
        for k in KEYS:
            assert rel(g[k], w[k]) < TOL, (j, k, rel(g[k], w[k]))
        if n_chains >= 2:
            assert rel(g["Rhat"], w["Rhat"]) < TOL, (j, rel(g["Rhat"], w["Rhat"]))
        else:
            assert np.all(np.isnan(g["Rhat"]))
    eng.close()
    return got


def test_exact_64x64_three_chains(sbd, cman):
    _exact(sbd, _crop(cman, (64, 64)), 3, 7)


def test_exact_243x375_two_chains_odd_pixels(sbd, boat):
    """odd pixel count: the scalar path of k_langevin; partial edge blocks at every level"""
    _exact(sbd, _crop(boat, (243, 375)), 2, 5)


def test_exact_120x200_blocks_larger_than_the_image(sbd, cman):
    got = _exact(sbd, _crop(cman, (120, 200)), 2, 7)
    assert got[6]["mean"].shape == (2, 4)


def test_existing_outputs_untouched(sbd, cman):
    x = _crop(cman, (96, 128))
    eng = sbd.Engine(96, 128, 7, sbd.MOFFAT, 0.0, max_batch=2)
    y, mk = _problem(sbd, eng, x, 4, 12, n_chains=2)
    a = eng.sapg(y, mk(post_mean=1), want_X_mean=True)
    b = eng.sapg(y, mk(post_mean=1), want_X_mean=True, post_levels=4)
    assert "posterior" not in a
    for k in TRAJ + ("X_mean", "X_last", "X_warm", "logPiTrace_WU"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k            # (tol_* start with NaN, as the reference)
    assert np.array_equal(b["posterior"][0]["mean"], a["X_mean"])
    # statistics without post_mean: no X_mean asked for, the same statistics
    c = eng.sapg(y, mk(post_mean=0), want_X_mean=True, post_levels=4)
    assert not np.any(c["X_mean"]) and "X_mean" in c
    for j in range(4):
        for k in ("mean", "within", "between"):
            assert np.array_equal(b["posterior"][j][k], c["posterior"][j][k])
    eng.close()


def test_graph_eager_and_serial_streams_identical(sbd, cman):
    x = _crop(cman, (128, 96))
    eng = sbd.Engine(128, 96, 7, sbd.MOFFAT, 0.0, max_batch=2)
    y, mk = _problem(sbd, eng, x, 3, 12, n_chains=2)
    outs = [eng.sapg(y, mk(use_graph=1), post_levels=5), eng.sapg(y, mk(use_graph=0), post_levels=5)]
    eng.set_option("overlap", 0)
    outs.append(eng.sapg(y, mk(use_graph=0), post_levels=5))
    outs.append(eng.sapg(y, mk(use_graph=1), post_levels=5))
    eng.set_option("overlap", -1)
    for o in outs[1:]:
        for j in range(5):
            for k in ("mean", "within", "between"):
                assert np.array_equal(o["posterior"][j][k], outs[0]["posterior"][j][k]), (j, k)
    eng.close()


class NoiseTape:
    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.tape = []
        self.record = False

    def __call__(self, shape):
        z = self.rng.standard_normal(shape)
        if self.record:
            self.tape.append(z)
        return z


@pytest.mark.parametrize("model", [0, 2])
def test_against_the_oracle_sapg(sbd, cman, model):
    """var / std at the pixel scale and at s = 4 against the oracle SAPG's samples (gradF spy), same noise tape"""
    import oracle as O
    from oracle import posterior as OP
    x = cman[64:128, 96:160].copy()
    tape = NoiseTape(40 + model)
    if model == 0:
        y, op, c = O.operators.setup_demo(0, x, tape, samples=14, warmup=4, burnIn=6, fix_w1=0, fix_w2=0)
    else:
        y, op = O.operators.setup_demo(2, x, tape, samples=14, warmup=4, burnIn=6)
    tape.record = True
    Xs = []
    op2 = dict(op)
    gradF = op["gradF"]

    def spy(X, *a):
        Xs.append(X.copy())
        return gradF(X, *a)

    op2["gradF"] = spy
    if model == 0:
        r = O.sapg.SAPG_algorithm_Guassian(y, op2, c, tape)[-1]
    else:
        r = O.sapg.SAPG_algorithm_laplace(y, op2, tape)[-1]
    noise = np.stack(tape.tape)[:, None]
    if model == 0:
        g = sbd.SAPG_algorithm_Guassian(y, op, c, noise=noise, post_levels=3)[-1]
        last = r["Xlast_sample"]
    else:
        g = sbd.SAPG_algorithm_laplace(y, op, noise=noise, post_levels=3)[-1]
        last = r["X_sample"]
    W, S, B = op["warmup"], op["samples"], op["burnIn"]
    main = Xs[(W - 1):] + [last]                      # X_1 .. X_S of the main loop
    want = OP.stats(np.stack(main[B:S])[:, None], 3)
    for j in (0, 2):
        for k in ("var", "std"):
            assert rel(g["posterior"][j][k], want[j][k]) < TRAJ_TOL, (j, k)
    assert rel(g["posteriorvar"], want[0]["var"]) < TRAJ_TOL and rel(g["posteriorstd"], want[0]["std"]) < TRAJ_TOL
    assert np.all(np.isnan(g["Rhat"]))               # one chain


def test_large_shape_2160x3840(sbd, boat):
    from oracle import posterior as OP
    x = _crop(boat, (2160, 3840))
    eng = sbd.Engine(2160, 3840, 7, sbd.MOFFAT, 0.0, max_batch=2)
    burnIn, extra, L = 2, 3, 7
    y, mk = _problem(sbd, eng, x, burnIn, burnIn + extra, n_chains=2)
    runs = [eng.sapg(y, mk(samples=burnIn + k), want_X_warm=False, post_levels=L if k == extra else 0)
            for k in range(1, extra + 1)]
    samples = np.stack([r["X_last"] for r in runs])
    rng = np.random.default_rng(5)
    for j in range(L):
        s = 1 << j
        g = runs[-1]["posterior"][j]
        bx, by = g["mean"].shape
        assert (bx, by) == (-(-2160 // s), -(-3840 // s))
        I = np.append(rng.integers(0, bx, 255), bx - 1)     # a seeded subset of blocks, with the corner one
        J = np.append(rng.integers(0, by, 255), by - 1)
        # block means of the chosen blocks (slicing keeps partial edge blocks partial), then the oracle on them
        v = np.stack([samples[:, :, i * s:(i + 1) * s, jj * s:(jj + 1) * s].mean(axis=(2, 3)) for i, jj in zip(I, J)],
                     axis=-1)[..., None]                     # [extra, C, blocks, 1]
        w = OP.stats(v, 1)[0]
        for k in KEYS:
            assert rel(g[k][I, J], w[k][:, 0]) < TOL, (j, k, rel(g[k][I, J], w[k][:, 0]))
        assert rel(g["Rhat"][I, J], w["Rhat"][:, 0]) < TOL
    eng.close()


def test_errors_and_launch_count(sbd, cman):
    from sbd_b200 import SbdError, lib
    x = _crop(cman, (64, 64))
    eng = sbd.Engine(64, 64, 7, sbd.MOFFAT, 0.0, max_batch=1)
    y, mk = _problem(sbd, eng, x, 3, 8)
    with pytest.raises(SbdError) as e:                 # before any run with statistics
        eng.posterior_stats(0)
    assert e.value.code == -1 and "no statistics" in e.value.msg
    with pytest.raises(SbdError) as e:
        eng.set_posterior(8)
    assert e.value.code == -1
    with pytest.raises(SbdError) as e:                 # burnIn = 0: the first sample would be divided by 2
        eng.sapg(y, mk(burnIn=0), post_levels=2)
    assert e.value.code == -1 and "burnIn" in e.value.msg
    r = eng.sapg(y, mk(), post_levels=2)
    assert [p["n"] for p in r["posterior"]] == [5, 5]
    with pytest.raises(SbdError) as e:                 # level >= L
        eng.posterior_stats(2)
    assert e.value.code == -1
    eng.posterior_stats(1)
    # samples <= burnIn: n = 0, zero arrays
    z = eng.sapg(y, mk(samples=3), post_levels=2)["posterior"]
    assert z[0]["n"] == 0 and not np.any(z[0]["mean"]) and not np.any(z[1]["within"])
    # after switching the statistics off the iteration launches what a context that never had them launches
    off = eng.sapg(y, mk(use_graph=0))["launches_main"]
    fresh = sbd.Engine(64, 64, 7, sbd.MOFFAT, 0.0, max_batch=1)
    assert fresh.sapg(y, mk(use_graph=0))["launches_main"] == off
    with pytest.raises(SbdError):                      # no run with statistics on that context
        fresh.posterior_stats(0)
    on = eng.sapg(y, mk(use_graph=0), post_levels=3)["launches_main"]
    assert on == off + (8 - 1)                         # one k_post_blocks per main-loop iteration
    assert lib.sbd_set_posterior(eng._h, 0) == 0
    fresh.close()
    eng.close()


def test_sapg_wrappers_keep_the_reference_field_set(sbd, cman):
    import oracle as O
    x = cman[64:128, 96:160].copy()
    tape = NoiseTape(50)
    y, op, c = O.operators.setup_demo(0, x, tape, samples=8, warmup=3, burnIn=4, fix_w1=0, fix_w2=0)
    a = sbd.SAPG_algorithm_Guassian(y, op, c, n_chains=2)[-1]
    b = sbd.SAPG_algorithm_Guassian(y, op, c, n_chains=2, post_levels=2)[-1]
    assert set(b) - set(a) == {"posterior", "posteriorvar", "posteriorstd", "Rhat"}
    assert np.all(np.isfinite(b["Rhat"])) and b["posterior"][1]["scale"] == 2
    assert b["posterior"][0]["n"] == 4 and b["posterior"][0]["chains"] == 2


def test_demo_run_batch_saves_std_and_rhat(cman, tmp_path):
    from sbd_b200 import demo
    x = cman[64:128, 96:160].copy()
    out = demo.run_batch(0, {"crop": x}, bsnrs=(30,), out_dir=str(tmp_path), samples=8, warmup=3, burnIn=4,
                         map_estimate=False, n_chains=2, post_levels=2, fix_w1=0, fix_w2=0)
    res = out[("crop", 30)]
    assert res["posteriorstd"].shape == x.shape
    z = np.load(tmp_path / "gaussian_crop_bsnr30.npz")
    assert z["posterior_std_s1"].shape == (64, 64) and z["Rhat_s2"].shape == (32, 32)
    assert np.array_equal(z["posterior_std_s1"], res["posteriorstd"])


# ---------------------------------------------------------------- MEX
def test_mex_gateway_posterior(cman):
    sys.path.insert(0, os.path.join(ROOT, "tests", "mexrt"))
    import runtime as mex
    from oracle import posterior as OP
    x = cman[64:128, 96:160].copy()
    rng = np.random.default_rng(9)
    y = x + 3.0 * rng.standard_normal(x.shape)
    P = dict(samples=8, warmup=3, burnIn=4, n_chains=2, gam=0.5, lamb=1.0, prox_lambda=1.0, th_init=0.01, min_th=1e-3,
             max_th=1.0, c_theta=0.01, psi_init=[0.5, 0.3], psi_min=[0.1, 0.1], psi_max=[1.0, 1.0], c_psi=[10.0, 10.0],
             psi_fixed=[0.4, 0.3], psi_true=[0.4, 0.3], fix_psi=[0.0, 0.0], sigma2_init=9.0, sigma2_min=1.0,
             sigma2_max=100.0, c_sigma2=1000.0, sigma2_fixed=9.0, err_psf_lag=1, d_scale=1.0, d_exp=0.8, seed=3)
    plain = mex.call_mex("sapg", y, None, None, 0, 7, 0.0, P, None)[0]
    assert "posterior" not in plain
    r = mex.call_mex("sapg", y, None, None, 0, 7, 0.0, dict(P, post_levels=3), None)[0]
    assert set(r) - set(plain) == {"posterior"}
    assert sorted(r["posterior"]) == ["s1", "s2", "s4"]
    for k in plain:
        if k != "seconds":
            assert np.array_equal(plain[k], r[k], equal_nan=True), k
    for j, name in enumerate(("s1", "s2", "s4")):
        e = r["posterior"][name]
        assert float(e["scale"]) == 1 << j and float(e["n"]) == 4 and float(e["chains"]) == 2
        var, std, rhat = OP.moments(e["mean"], e["within"], e["between"], 4, 2)
        for got, want in ((e["var"], var), (e["std"], std), (e["Rhat"], rhat)):
            assert np.allclose(got, want, rtol=TOL, atol=0, equal_nan=True)
    # the cached context has its statistics switched off again
    again = mex.call_mex("sapg", y, None, None, 0, 7, 0.0, P, None)[0]
    assert "posterior" not in again


# ---------------------------------------------------------------- 2 GPUs
MERGE_WORKER = textwrap.dedent("""
    import os, sys, pickle
    import numpy as np
    import torch, torch.distributed as dist
    sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
    import sbd_b200
    from sbd_b200 import host as H
    from test_gpu_posterior import _problem
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo")
    total, per = 4, 4 // world
    x = np.load(sys.argv[2])
    eng = sbd_b200.Engine(x.shape[0], x.shape[1], 7, H.MOFFAT, 0.0, total, rank)
    y, mk = _problem(sbd_b200, eng, x, 3, 9)
    shard = sbd_b200.ChainShard(total, world, rank)
    shard.init_engine_comm(eng)
    prm = mk(); prm.n_chains = per; prm.chain_offset = shard.chain_offset; prm.total_chains = total
    merged = shard.combine_posterior(eng.sapg(y, prm, post_levels=4)["posterior"])
    sbd_b200._lib.lib.sbd_comm_destroy(eng._h)
    if rank == 0:
        prm = mk(); prm.n_chains = total; prm.total_chains = total
        ref = eng.sapg(y, prm, post_levels=4)["posterior"]
        ok = all(np.linalg.norm(m[k] - r[k]) <= 1e-12 * np.linalg.norm(r[k])
                 for m, r in zip(merged, ref) for k in ("mean", "within", "between", "var", "std", "Rhat"))
        print("merged:", ok and all(m["chains"] == 4 for m in merged))
    dist.barrier()
    dist.destroy_process_group()
    eng.close()
""")


def test_two_gpus_merged_equal_one_gpu(cman, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    worker = tmp_path / "worker.py"
    worker.write_text(MERGE_WORKER)
    np.save(tmp_path / "x.npy", _crop(cman, (96, 128)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29613", str(worker), ROOT, str(tmp_path / "x.npy")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "merged: True" in r.stdout
