"""GPU tests of the posterior quantiles (include/sbd.h sbd_set_posterior_quantiles / sbd_posterior_quantiles, DESIGN.md
"Credible intervals and the median"): bitwise against tests/posterior_quantile_oracle.py on the device's own samples
at every level, everything else bitwise unchanged with one more launch per main-loop iteration, graph / eager /
serial streams bitwise identical, a large shape, the error paths, the SAPG wrappers and demo, and the MEX gateway."""
import os
import sys

import numpy as np
import pytest

import posterior_quantile_oracle as PQ
from conftest import ROOT
from test_gpu_posterior import _crop, _problem, TRAJ

pytestmark = pytest.mark.gpu

QKEYS = ("lower", "median", "upper", "ci_width")
STATS = ("mean", "within", "between", "var", "std", "Rhat")
DIAG = ("batch_mean", "batch_within", "batch_between", "half_mean", "half_within", "half_between", "ESS", "MCSE",
        "Rhat_split")


@pytest.fixture(scope="module")
def sbd():
    import sbd_b200
    return sbd_b200


def _exact(sbd, x, n_chains, levels, cases, burnIn=2):
    """Runs with samples = burnIn+1 .. burnIn+extra return the exact device samples X_ii as their last samples (they
    are prefixes of one another); `cases` is a list of (k, alpha, post_batch): the run with n = k window samples
    repeated with quantiles, compared bitwise with the oracle fed the first k samples."""
    extra = max(c[0] for c in cases)
    eng = sbd.Engine(x.shape[0], x.shape[1], 7, sbd.MOFFAT, 0.0, max_batch=n_chains)
    y, mk = _problem(sbd, eng, x, burnIn, burnIn + extra, n_chains=n_chains)
    runs = [eng.sapg(y, mk(samples=burnIn + k), want_X_warm=False) for k in range(1, extra + 1)]
    samples = np.stack([r["X_last"] for r in runs])                        # [extra, C, rows, cols]
    for k, alpha, b in cases:
        got = eng.sapg(y, mk(samples=burnIn + k), want_X_warm=False, post_levels=levels, post_batch=b, post_ci=alpha)
        assert np.array_equal(got["X_last"], runs[k - 1]["X_last"])
        want = PQ.quantiles(samples[:k], levels, alpha)
        assert len(got["posterior"]) == levels
        for j, (g, w) in enumerate(zip(got["posterior"], want)):
            assert g["ci_alpha"] == alpha and g["ci_count"] == w["count"] == n_chains * k
            assert g["median"].shape == w["median"].shape == (-(-x.shape[0] >> j), -(-x.shape[1] >> j))
            for key in QKEYS:
                assert np.array_equal(g[key], w[key], equal_nan=True), (k, alpha, j, key)
    eng.close()


def test_exact_64x64_three_chains(sbd, cman):
    # N = 6 < 9 (interpolated), N = 9 exactly (the sorted markers), N = 51 (marker adjustments)
    _exact(sbd, _crop(cman, (64, 64)), 3, 7, [(2, 0.1, 0), (3, 0.05, 0), (17, 0.1, 0), (17, 0.05, 0)])


def test_exact_243x375_two_chains_odd_pixels(sbd, boat):
    """odd pixel count and partial edge blocks at every level"""
    _exact(sbd, _crop(boat, (243, 375)), 2, 5, [(12, 0.1, 0)])


def test_exact_one_chain(sbd, cman):
    """the reference's configuration"""
    _exact(sbd, _crop(cman, (96, 128)), 1, 3, [(30, 0.1, 0)])


def test_exact_with_diagnostics(sbd, cman):
    """k_post_blocks<true, true>: the block means with the diagnostics on as well"""
    _exact(sbd, _crop(cman, (80, 72)), 2, 4, [(10, 0.1, -1), (10, 0.2, 3)])


def test_quantiles_leave_everything_else_unchanged(sbd, cman):
    x = _crop(cman, (96, 128))
    eng = sbd.Engine(96, 128, 7, sbd.MOFFAT, 0.0, max_batch=2)
    samples = 15
    y, mk = _problem(sbd, eng, x, 4, samples, n_chains=2)
    for graph in (0, 1):
        for b in (0, -1):
            a = eng.sapg(y, mk(post_mean=1, use_graph=graph), want_X_mean=True, post_levels=4, post_batch=b)
            q = eng.sapg(y, mk(post_mean=1, use_graph=graph), want_X_mean=True, post_levels=4, post_batch=b,
                         post_ci=0.1)
            assert not any(k in p for p in a["posterior"] for k in QKEYS)
            for k in TRAJ + ("X_mean", "X_last", "X_warm", "logPiTrace_WU"):
                assert np.array_equal(a[k], q[k], equal_nan=True), k
            for pa, pq in zip(a["posterior"], q["posterior"]):
                for k in STATS + ("scale", "n", "chains") + (DIAG if b else ()):
                    assert np.array_equal(pa[k], pq[k], equal_nan=True), k
            assert q["launches_main"] == a["launches_main"] + (samples - 1), (graph, b)
    # L = 1: no block kernel, still exactly one more launch per iteration
    a = eng.sapg(y, mk(use_graph=0), post_levels=1)
    q = eng.sapg(y, mk(use_graph=0), post_levels=1, post_ci=0.1)
    assert q["launches_main"] == a["launches_main"] + (samples - 1)
    eng.close()


def test_graph_eager_and_serial_streams_identical(sbd, cman):
    x = _crop(cman, (128, 96))
    eng = sbd.Engine(128, 96, 7, sbd.MOFFAT, 0.0, max_batch=2)
    y, mk = _problem(sbd, eng, x, 3, 14, n_chains=2)
    outs = [eng.sapg(y, mk(use_graph=1), post_levels=5, post_ci=0.1),
            eng.sapg(y, mk(use_graph=0), post_levels=5, post_ci=0.1)]
    eng.set_option("overlap", 0)
    outs.append(eng.sapg(y, mk(use_graph=0), post_levels=5, post_ci=0.1))
    outs.append(eng.sapg(y, mk(use_graph=1), post_levels=5, post_ci=0.1))
    eng.set_option("overlap", -1)
    for o in outs[1:]:
        for j in range(5):
            for k in QKEYS:
                assert np.array_equal(o["posterior"][j][k], outs[0]["posterior"][j][k]), (j, k)
    eng.close()


def test_large_shape_2160x3840(sbd, boat):
    x = _crop(boat, (2160, 3840))
    eng = sbd.Engine(2160, 3840, 7, sbd.MOFFAT, 0.0, max_batch=2)
    burnIn, extra, L, alpha = 2, 6, 7, 0.1                  # N = 12: the insertion phase and three P^2 updates
    y, mk = _problem(sbd, eng, x, burnIn, burnIn + extra, n_chains=2)
    runs = [eng.sapg(y, mk(samples=burnIn + k), want_X_warm=False, post_levels=L if k == extra else 0,
                     post_ci=alpha if k == extra else 0.0) for k in range(1, extra + 1)]
    samples = np.stack([r["X_last"] for r in runs])
    got = runs[-1]["posterior"]
    for j in (0, 6):
        w = PQ.p2(samples if j == 0 else PQ.block_means_nested(samples, 1 << j), alpha)
        assert got[j]["ci_count"] == w["count"] == 12
        for k in ("lower", "median", "upper"):
            assert np.array_equal(got[j][k], w[k]), (j, k)
    assert got[6]["median"].shape == (34, 60)
    eng.close()


def test_errors(sbd, cman):
    import ctypes as C
    from sbd_b200 import SbdError, lib
    from sbd_b200._lib import sbd_traces
    x = _crop(cman, (64, 64))
    eng = sbd.Engine(64, 64, 7, sbd.MOFFAT, 0.0, max_batch=2)
    y, mk = _problem(sbd, eng, x, 3, 8)
    for bad in (float("nan"), -0.1, 1.0, 1.5):
        with pytest.raises(SbdError) as e:
            eng.set_posterior_quantiles(bad)
        assert e.value.code == -1 and "alpha" in e.value.msg
    with pytest.raises(SbdError) as e:                 # before any run with quantiles
        eng.posterior_quantiles(0)
    assert e.value.code == -1 and "no quantiles" in e.value.msg
    with pytest.raises(SbdError) as e:                 # quantiles without the statistics
        eng.sapg(y, mk(), post_ci=0.1)
    assert e.value.code == -1 and "sbd_set_posterior" in e.value.msg
    eng.sapg(y, mk(), post_levels=2)                   # statistics only: no quantiles to read
    with pytest.raises(SbdError) as e:
        eng.posterior_quantiles(0)
    assert e.value.code == -1
    r = eng.sapg(y, mk(), post_levels=2, post_ci=0.1)["posterior"]
    assert r[1]["ci_count"] == 5 and r[1]["median"].shape == (32, 32)
    with pytest.raises(SbdError) as e:                 # level >= L
        eng.posterior_quantiles(2)
    assert e.value.code == -1 and "level" in e.value.msg
    eng.posterior_quantiles(1)
    # samples <= burnIn: no values, NaN (not an error)
    z = eng.sapg(y, mk(samples=3), post_levels=2, post_ci=0.1)["posterior"]
    for d in z:
        assert d["ci_count"] == 0 and all(np.all(np.isnan(d[k])) for k in QKEYS)
    # C*n >= 2^31: the int32 marker positions would overflow; refused before any work
    prm = mk(samples=(1 << 30) + 10)
    prm.n_chains = prm.total_chains = 2
    yb = np.asfortranarray(y)
    assert lib.sbd_set_posterior(eng._h, 1) == 0 and lib.sbd_set_posterior_quantiles(eng._h, 0.1) == 0
    tr = sbd_traces()
    rc = lib.sbd_sapg_run(eng._h, yb.ctypes.data_as(C.POINTER(C.c_double)), None, None, C.byref(prm), None,
                          C.byref(tr))
    assert rc == -1 and "2^31" in lib.sbd_last_error(eng._h).decode()
    # Engine.sapg leaves the requests off
    assert lib.sbd_set_posterior_quantiles(eng._h, 0.0) == 0 and lib.sbd_set_posterior(eng._h, 0) == 0
    plain = eng.sapg(y, mk(), post_levels=1)["posterior"][0]
    assert "median" not in plain
    eng.close()


def test_sapg_wrappers_and_demo(sbd, cman, tmp_path):
    import oracle as O
    from sbd_b200 import demo
    from test_gpu_posterior import NoiseTape
    x = cman[64:128, 96:160].copy()
    y, op, c = O.operators.setup_demo(0, x, NoiseTape(50), samples=16, warmup=3, burnIn=4, fix_w1=0, fix_w2=0)
    a = sbd.SAPG_algorithm_Guassian(y, op, c, n_chains=2, post_levels=2)[-1]
    b = sbd.SAPG_algorithm_Guassian(y, op, c, n_chains=2, post_levels=2, post_ci=0.1)[-1]
    assert set(b) - set(a) == {"posteriormedian", "CI_lower", "CI_upper"}
    assert np.array_equal(b["posteriormedian"], b["posterior"][0]["median"]) and b["CI_lower"].shape == x.shape
    assert np.all(b["CI_lower"] <= b["posteriormedian"]) and np.all(b["posteriormedian"] <= b["CI_upper"])
    assert np.all(b["CI_lower"] >= 0)                  # the MYULA fold: unlike mean - z*std, never below zero
    out = demo.run_batch(0, {"crop": x}, bsnrs=(30,), out_dir=str(tmp_path), samples=16, warmup=3, burnIn=4,
                         map_estimate=False, n_chains=2, post_levels=2, post_ci=0.1, fix_w1=0, fix_w2=0)
    res = out[("crop", 30)]
    z = np.load(tmp_path / "gaussian_crop_bsnr30.npz")
    assert z["CI_width_s1"].shape == (64, 64) and z["CI_width_s2"].shape == (32, 32)
    assert np.array_equal(z["CI_width_s1"], res["CI_upper"] - res["CI_lower"])


def test_mex_gateway_quantiles(cman):
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
    extra = {"ci_alpha", "ci_count", "lower", "median", "upper", "ci_width"}
    for batch in (0, -1):
        r = mex.call_mex("sapg", y, None, None, 0, 7, 0.0, dict(P, post_ci=0.1, post_batch=batch), None)[0]
        for name in ("s1", "s2", "s4"):
            p, e = plain["posterior"][name], r["posterior"][name]
            assert extra <= set(e) and set(p) <= set(e)
            assert np.asarray(e["ci_alpha"]).item() == 0.1 and np.asarray(e["ci_count"]).item() == 18
            assert np.array_equal(e["ci_width"], np.asarray(e["upper"]) - np.asarray(e["lower"]))
            assert np.all(np.asarray(e["lower"]) <= np.asarray(e["median"]))
            assert np.all(np.asarray(e["median"]) <= np.asarray(e["upper"]))
            for k in p:
                assert np.array_equal(p[k], e[k], equal_nan=True), (name, k)
    # the cached context has the request switched off again
    again = mex.call_mex("sapg", y, None, None, 0, 7, 0.0, P, None)[0]
    assert set(again["posterior"]["s1"]) == set(plain["posterior"]["s1"])
