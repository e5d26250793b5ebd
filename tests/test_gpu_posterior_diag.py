"""GPU tests of the posterior diagnostics (include/sbd.h sbd_set_posterior_diagnostics / sbd_posterior_diagnostics,
DESIGN.md "Posterior statistics"): exact against tests/posterior_diag_oracle.py on the device's own samples, everything else
bitwise unchanged, graph / eager / serial streams bitwise identical, a large shape, a long single chain, the error
paths, the SAPG wrappers and demo, the MEX gateway and a 2-GPU merge."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import posterior_diag_oracle as PD
from conftest import rel, ROOT
from test_gpu_posterior import _crop, _problem, TRAJ

pytestmark = pytest.mark.gpu

TOL = 1e-12             # sufficient statistics
DTOL = 1e-10            # ESS, MCSE, Rhat_split
SUFF = ("batch_mean", "batch_within", "batch_between", "half_mean", "half_within", "half_between")
DERIVED = ("ESS", "MCSE", "Rhat_split")
STATS = ("mean", "within", "between", "var", "std", "Rhat")


@pytest.fixture(scope="module")
def sbd():
    import sbd_b200
    return sbd_b200


def _close(got, want, tol):
    """relative 2-norm error over the finite entries; NaN exactly where the oracle has NaN"""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    return rel(got[ok], want[ok]) < tol if ok.any() else True


def _exact(sbd, x, n_chains, levels, cases, burnIn=2):
    """Runs with samples = burnIn+1 .. burnIn+extra return the exact device samples X_ii as their last samples (they
    are prefixes of one another); `cases` is a list of (k, b): the run with n = k window samples repeated with
    post_batch b, its diagnostics compared with tests/posterior_diag_oracle.py on the first k samples."""
    extra = max(k for k, _ in cases)
    eng = sbd.Engine(x.shape[0], x.shape[1], 7, sbd.MOFFAT, 0.0, max_batch=n_chains)
    y, mk = _problem(sbd, eng, x, burnIn, burnIn + extra, n_chains=n_chains)
    runs = [eng.sapg(y, mk(samples=burnIn + k), want_X_warm=False) for k in range(1, extra + 1)]
    samples = np.stack([r["X_last"] for r in runs])                        # [extra, C, rows, cols]
    for k, b in cases:
        got = eng.sapg(y, mk(samples=burnIn + k), want_X_warm=False, post_levels=levels, post_batch=b)
        assert np.array_equal(got["X_last"], runs[k - 1]["X_last"])
        want = PD.diagnostics(samples[:k], levels, b)
        for j, (g, w) in enumerate(zip(got["posterior"], want)):
            assert (g["batch_len"], g["n_batches"], g["half_n"]) == (w["batch_len"], w["n_batches"], w["half_n"])
            assert g["batch_mean"].shape == w["batch_mean"].shape
            for key in SUFF:
                assert rel(g[key], w[key]) < TOL, (k, b, j, key, rel(g[key], w[key]))
            for key in DERIVED:
                assert _close(g[key], w[key], DTOL), (k, b, j, key)
    eng.close()


def test_exact_64x64_three_chains(sbd, cman):
    # n = 7 (odd), b = 2: B*b = 6 < n; automatic b = 2; n = 6 with b = 4 (B = 1) and b = 1; b > n: B = 0
    _exact(sbd, _crop(cman, (64, 64)), 3, 7, [(7, 2), (7, -1), (6, 4), (6, 1), (5, 9)])


def test_exact_243x375_two_chains_odd_pixels(sbd, boat):
    """odd pixel count: the scalar path of k_langevin; partial edge blocks at every level"""
    _exact(sbd, _crop(boat, (243, 375)), 2, 5, [(8, 3), (8, -1), (9, -1), (5, 2)])


def test_diagnostics_leave_everything_else_unchanged(sbd, cman):
    x = _crop(cman, (96, 128))
    eng = sbd.Engine(96, 128, 7, sbd.MOFFAT, 0.0, max_batch=2)
    y, mk = _problem(sbd, eng, x, 4, 15, n_chains=2)
    for graph in (0, 1):
        a = eng.sapg(y, mk(post_mean=1, use_graph=graph), want_X_mean=True, post_levels=4)
        b = eng.sapg(y, mk(post_mean=1, use_graph=graph), want_X_mean=True, post_levels=4, post_batch=-1)
        assert not any(k in p for p in a["posterior"] for k in SUFF + DERIVED)
        for k in TRAJ + ("X_mean", "X_last", "X_warm", "logPiTrace_WU"):
            assert np.array_equal(a[k], b[k], equal_nan=True), k
        for pa, pb in zip(a["posterior"], b["posterior"]):
            for k in STATS + ("scale", "n", "chains"):
                assert np.array_equal(pa[k], pb[k], equal_nan=True), k
        assert a["launches_main"] == b["launches_main"]
    eng.close()


def test_graph_eager_and_serial_streams_identical(sbd, cman):
    x = _crop(cman, (128, 96))
    eng = sbd.Engine(128, 96, 7, sbd.MOFFAT, 0.0, max_batch=2)
    y, mk = _problem(sbd, eng, x, 3, 14, n_chains=2)
    outs = [eng.sapg(y, mk(use_graph=1), post_levels=5, post_batch=3),
            eng.sapg(y, mk(use_graph=0), post_levels=5, post_batch=3)]
    eng.set_option("overlap", 0)
    outs.append(eng.sapg(y, mk(use_graph=0), post_levels=5, post_batch=3))
    outs.append(eng.sapg(y, mk(use_graph=1), post_levels=5, post_batch=3))
    eng.set_option("overlap", -1)
    for o in outs[1:]:
        for j in range(5):
            for k in SUFF:
                assert np.array_equal(o["posterior"][j][k], outs[0]["posterior"][j][k]), (j, k)
    eng.close()


def test_large_shape_2160x3840(sbd, boat):
    x = _crop(boat, (2160, 3840))
    eng = sbd.Engine(2160, 3840, 7, sbd.MOFFAT, 0.0, max_batch=2)
    burnIn, extra, L, bl = 2, 5, 7, 2
    y, mk = _problem(sbd, eng, x, burnIn, burnIn + extra, n_chains=2)
    runs = [eng.sapg(y, mk(samples=burnIn + k), want_X_warm=False, post_levels=L if k == extra else 0,
                     post_batch=bl if k == extra else 0) for k in range(1, extra + 1)]
    samples = np.stack([r["X_last"] for r in runs])
    rng = np.random.default_rng(5)
    for j in range(L):
        s = 1 << j
        g = runs[-1]["posterior"][j]
        bx, by = g["batch_mean"].shape
        assert (bx, by) == (-(-2160 // s), -(-3840 // s))
        assert (g["batch_len"], g["n_batches"], g["half_n"]) == (2, 2, 2)
        I = np.append(rng.integers(0, bx, 255), bx - 1)     # a seeded subset of blocks, with the corner one
        J = np.append(rng.integers(0, by, 255), by - 1)
        v = np.stack([samples[:, :, i * s:(i + 1) * s, jj * s:(jj + 1) * s].mean(axis=(2, 3)) for i, jj in zip(I, J)],
                     axis=-1)[..., None]                     # [extra, C, blocks, 1]
        w = PD.diagnostics(v, 1, bl)[0]
        for k in SUFF:
            assert rel(g[k][I, J], w[k][:, 0]) < TOL, (j, k, rel(g[k][I, J], w[k][:, 0]))
        for k in DERIVED:
            assert rel(g[k][I, J], w[k][:, 0]) < DTOL, (j, k)
    eng.close()


def test_one_chain_split_rhat_and_ess(sbd, cman):
    """the reference's configuration: one chain, where the classic Rhat is NaN"""
    eng = sbd.Engine(256, 256, 7, sbd.MOFFAT, 0.0, max_batch=1)
    y, mk = _problem(sbd, eng, cman, 100, 400)
    p = eng.sapg(y, mk(), want_X_warm=False, post_levels=3, post_batch=-1)["posterior"]
    assert (p[0]["batch_len"], p[0]["n_batches"], p[0]["half_n"]) == (17, 17, 150)
    for d in p:
        assert np.all(np.isnan(d["Rhat"]))
        for k in ("ESS", "MCSE", "Rhat_split"):
            assert np.all(np.isfinite(d[k])) and np.all(d[k] > 0), k
    eng.close()


def test_errors(sbd, cman):
    from sbd_b200 import SbdError, lib
    x = _crop(cman, (64, 64))
    eng = sbd.Engine(64, 64, 7, sbd.MOFFAT, 0.0, max_batch=1)
    y, mk = _problem(sbd, eng, x, 3, 8)
    with pytest.raises(SbdError) as e:
        eng.set_posterior_diagnostics(-2)
    assert e.value.code == -1 and "batch_len" in e.value.msg
    with pytest.raises(SbdError) as e:                 # before any run with diagnostics
        eng.posterior_diagnostics(0)
    assert e.value.code == -1 and "no diagnostics" in e.value.msg
    with pytest.raises(SbdError) as e:                 # diagnostics without the statistics
        eng.sapg(y, mk(), post_batch=-1)
    assert e.value.code == -1 and "sbd_set_posterior" in e.value.msg
    eng.sapg(y, mk(), post_levels=2)                   # statistics only: no diagnostics to read
    with pytest.raises(SbdError) as e:
        eng.posterior_diagnostics(0)
    assert e.value.code == -1
    r = eng.sapg(y, mk(), post_levels=2, post_batch=2)["posterior"]
    assert (r[0]["batch_len"], r[0]["n_batches"], r[0]["half_n"]) == (2, 2, 2)
    with pytest.raises(SbdError) as e:                 # level >= L
        eng.posterior_diagnostics(2)
    assert e.value.code == -1
    eng.posterior_diagnostics(1)
    # b > n: no batches, NaN ESS / MCSE, not an error
    z = eng.sapg(y, mk(), post_levels=2, post_batch=6)["posterior"]
    for d in z:
        assert d["n_batches"] == 0 and not np.any(d["batch_within"]) and not np.any(d["batch_mean"])
        assert np.all(np.isnan(d["ESS"])) and np.all(np.isnan(d["MCSE"])) and np.all(np.isfinite(d["Rhat_split"]))
    # Engine.sapg leaves both requests off
    assert lib.sbd_set_posterior_diagnostics(eng._h, 0) == 0
    plain = eng.sapg(y, mk(), post_levels=1)["posterior"][0]
    assert "ESS" not in plain
    eng.close()


def test_sapg_wrappers_and_demo(sbd, cman, tmp_path):
    import oracle as O
    from sbd_b200 import demo
    from test_gpu_posterior import NoiseTape
    x = cman[64:128, 96:160].copy()
    y, op, c = O.operators.setup_demo(0, x, NoiseTape(50), samples=12, warmup=3, burnIn=4, fix_w1=0, fix_w2=0)
    a = sbd.SAPG_algorithm_Guassian(y, op, c, n_chains=2, post_levels=2)[-1]
    b = sbd.SAPG_algorithm_Guassian(y, op, c, n_chains=2, post_levels=2, post_batch=-1)[-1]
    assert set(b) - set(a) == {"ESS", "MCSE", "Rhat_split"}
    assert np.array_equal(b["ESS"], b["posterior"][0]["ESS"]) and b["MCSE"].shape == x.shape
    out = demo.run_batch(0, {"crop": x}, bsnrs=(30,), out_dir=str(tmp_path), samples=12, warmup=3, burnIn=4,
                         map_estimate=False, n_chains=2, post_levels=2, post_batch=-1, fix_w1=0, fix_w2=0)
    res = out[("crop", 30)]
    z = np.load(tmp_path / "gaussian_crop_bsnr30.npz")
    assert z["ESS_s1"].shape == (64, 64) and z["MCSE_s2"].shape == (32, 32) and z["Rhat_split_s2"].shape == (32, 32)
    assert np.array_equal(z["Rhat_split_s1"], res["Rhat_split"])


# ---------------------------------------------------------------- MEX
def test_mex_gateway_diagnostics(cman):
    sys.path.insert(0, os.path.join(ROOT, "tests", "mexrt"))
    import runtime as mex
    x = cman[64:128, 96:160].copy()
    rng = np.random.default_rng(9)
    y = x + 3.0 * rng.standard_normal(x.shape)
    P = dict(samples=13, warmup=3, burnIn=4, n_chains=2, gam=0.5, lamb=1.0, prox_lambda=1.0, th_init=0.01,
             min_th=1e-3, max_th=1.0, c_theta=0.01, psi_init=[0.5, 0.3], psi_min=[0.1, 0.1], psi_max=[1.0, 1.0],
             c_psi=[10.0, 10.0], psi_fixed=[0.4, 0.3], psi_true=[0.4, 0.3], fix_psi=[0.0, 0.0], sigma2_init=9.0,
             sigma2_min=1.0, sigma2_max=100.0, c_sigma2=1000.0, sigma2_fixed=9.0, err_psf_lag=1, d_scale=1.0,
             d_exp=0.8, seed=3, post_levels=3)
    plain = mex.call_mex("sapg", y, None, None, 0, 7, 0.0, P, None)[0]
    r = mex.call_mex("sapg", y, None, None, 0, 7, 0.0, dict(P, post_batch=-1), None)[0]
    extra = {"batch_mean", "batch_within", "batch_between", "half_mean", "half_within", "half_between", "batch_len",
             "n_batches", "half_n", "ESS", "MCSE", "Rhat_split"}
    for name in ("s1", "s2", "s4"):
        p, e = plain["posterior"][name], r["posterior"][name]
        assert set(p) == {"scale", "n", "chains", "mean", "within", "between", "var", "std", "Rhat"}
        assert set(e) - set(p) == extra
        assert [np.asarray(e[k]).item() for k in ("batch_len", "n_batches", "half_n")] == [3, 3, 4]
        for k in p:
            assert np.array_equal(p[k], e[k], equal_nan=True), (name, k)
        got = PD.diag_moments(e["var"], e["batch_within"], e["batch_between"], e["half_within"], e["half_between"],
                              9, 2, 3, 3, 4)
        for k, w in zip(DERIVED, got):
            assert np.allclose(e[k], w, rtol=1e-12, atol=0, equal_nan=True), (name, k)
    # the cached context has both requests switched off again
    again = mex.call_mex("sapg", y, None, None, 0, 7, 0.0, P, None)[0]
    assert set(again["posterior"]["s1"]) == set(plain["posterior"]["s1"])


# ---------------------------------------------------------------- 2 GPUs
MERGE_WORKER = textwrap.dedent("""
    import os, sys
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
    y, mk = _problem(sbd_b200, eng, x, 3, 12)
    shard = sbd_b200.ChainShard(total, world, rank)
    shard.init_engine_comm(eng)
    prm = mk(); prm.n_chains = per; prm.chain_offset = shard.chain_offset; prm.total_chains = total
    merged = shard.combine_posterior(eng.sapg(y, prm, post_levels=4, post_batch=-1)["posterior"])
    sbd_b200._lib.lib.sbd_comm_destroy(eng._h)
    if rank == 0:
        prm = mk(); prm.n_chains = total; prm.total_chains = total
        ref = eng.sapg(y, prm, post_levels=4, post_batch=-1)["posterior"]
        keys = ("batch_mean", "batch_within", "batch_between", "half_mean", "half_within", "half_between", "ESS",
                "MCSE", "Rhat_split")
        ok = all(np.linalg.norm(m[k] - r[k]) <= 1e-12 * np.linalg.norm(r[k]) for m, r in zip(merged, ref) for k in keys)
        print("merged:", ok and all(m["chains"] == 4 and m["n_batches"] == r["n_batches"] for m, r in zip(merged, ref)))
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
           "127.0.0.1", "--master-port", "29617", str(worker), ROOT, str(tmp_path / "x.npy")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "merged: True" in r.stdout
