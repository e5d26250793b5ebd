"""CPU tests of the posterior quantiles (DESIGN.md "Credible intervals and the median"; include/sbd.h
sbd_set_posterior_quantiles / sbd_posterior_quantiles): tests/posterior_quantile_oracle.py's block means against
oracle/posterior.py, its P^2 at N < 9, N = 9 and N = 0 against the definitions, its accuracy on i.i.d. and AR(1)
streams, ChainShard.combine_posterior with quantiles on one and on two gloo ranks, and the ctypes prototypes."""
import os
import sys

import numpy as np
import pytest
from scipy.stats import norm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import posterior_quantile_oracle as PQ  # noqa: E402
from oracle import posterior as OP  # noqa: E402


def _samples(S, C, rows, cols, seed):
    rng = np.random.default_rng(seed)
    return np.abs(100 + 20 * rng.standard_normal((S, C, rows, cols)))


def _ar1(n, C, rho, seed, E):
    """C independent stationary AR(1) chains per element, x_t = rho x_{t-1} + e_t, e ~ N(0, 1): marginal
    N(0, 1 / (1 - rho^2))"""
    rng = np.random.default_rng(seed)
    e = rng.standard_normal((n, C, E))
    x = np.empty_like(e)
    x[0] = e[0] / np.sqrt(1 - rho ** 2)
    for t in range(1, n):
        x[t] = rho * x[t - 1] + e[t]
    return x


@pytest.mark.parametrize("shape", [(37, 29), (7, 9), (64, 64), (130, 67)])
def test_nested_block_means_against_the_statistics_oracle(shape):
    x = _samples(2, 3, *shape, seed=shape[0])
    for j in range(7):
        s = 1 << j
        got = PQ.block_means_nested(x, s)
        want = OP.block_means(x, s)
        assert got.shape == want.shape == (2, 3, -(-shape[0] // s), -(-shape[1] // s))
        np.testing.assert_allclose(got, want, rtol=1e-13, atol=0)


@pytest.mark.parametrize("alpha", [0.1, 0.05, 0.5])
@pytest.mark.parametrize("S,C", [(1, 1), (2, 3), (1, 7), (4, 2), (8, 1)])
def test_fewer_than_nine_values_interpolate(S, C, alpha):
    x = _samples(S, C, 5, 4, seed=S * 10 + C)
    r = PQ.p2(x, alpha)
    N = S * C
    assert r["count"] == N < 9
    flat = x.reshape(N, -1)
    for key, p in (("lower", alpha / 2), ("median", 0.5), ("upper", 1 - alpha / 2)):
        got = r[key].reshape(-1)
        for e in range(flat.shape[1]):
            v = np.sort(flat[:, e])
            h = (N - 1) * p
            lo = int(np.floor(h))
            want = v[lo] if h == lo else v[lo] + (h - lo) * (v[lo + 1] - v[lo])
            assert got[e] == want, (key, e)
        np.testing.assert_allclose(got, np.quantile(flat, p, axis=0), rtol=1e-13)


def test_nine_values_are_the_sorted_markers():
    x = _samples(3, 3, 6, 5, seed=4)
    r = PQ.p2(x, 0.1)
    v = np.sort(x.reshape(9, 6, 5), axis=0)
    assert r["count"] == 9
    np.testing.assert_array_equal(r["q"], v)
    np.testing.assert_array_equal(r["n"][:, 0, 0], np.arange(1, 10))
    for key, i in (("lower", 2), ("median", 4), ("upper", 6)):
        np.testing.assert_array_equal(r[key], v[i])


def test_no_values_give_nan():
    r = PQ.quantiles(np.zeros((0, 2, 9, 7)), 3, 0.1)
    for j, d in enumerate(r):
        assert d["count"] == 0
        for k in ("lower", "median", "upper", "ci_width"):
            assert d[k].shape == (-(-9 // (1 << j)), -(-7 // (1 << j))) and np.all(np.isnan(d[k]))


def test_markers_stay_ordered_and_positions_consistent():
    x = _samples(60, 4, 8, 8, seed=12)
    r = PQ.p2(x, 0.1)
    assert np.all(np.diff(r["q"], axis=0) >= 0)
    assert np.all(np.diff(r["n"], axis=0) >= 1)
    assert np.all(r["n"][0] == 1) and np.all(r["n"][8] == 240)


def test_iid_normal_close_to_the_exact_sample_quantile():
    alpha = 0.1
    rng = np.random.default_rng(21)
    x = rng.standard_normal((5000, 1, 2000))
    r = PQ.p2(x, alpha)
    flat = x.reshape(5000, -1)
    for key, p in (("lower", alpha / 2), ("median", 0.5), ("upper", 1 - alpha / 2)):
        err = np.median(np.abs(r[key] - np.quantile(flat, p, axis=0)))
        assert err <= 0.01, (key, err)


@pytest.mark.parametrize("rho", [0.9, 0.99])
@pytest.mark.parametrize("C", [1, 8])
def test_ar1_within_the_monte_carlo_error_of_the_exact_quantile(rho, C):
    alpha = 0.1
    n = 4000 // C
    x = _ar1(n, C, rho, seed=int(rho * 100) + C, E=2000)
    r = PQ.p2(x, alpha)
    flat = x.reshape(n * C, -1)
    sd = 1 / np.sqrt(1 - rho ** 2)
    for key, p in (("lower", alpha / 2), ("median", 0.5), ("upper", 1 - alpha / 2)):
        true = norm.ppf(p) * sd
        exact = np.quantile(flat, p, axis=0)
        mc = np.median(np.abs(exact - true))
        assert np.median(np.abs(r[key] - true)) <= 1.25 * mc, (key, np.median(np.abs(r[key] - true)) / mc)
        assert np.median(np.abs(r[key] - exact)) <= 0.5 * mc, (key, np.median(np.abs(r[key] - exact)) / mc)


def _with_quantiles(x, levels, alpha):
    st = OP.stats(x, levels)
    for d, q in zip(st, PQ.quantiles(x, levels, alpha)):
        d.update(ci_alpha=alpha, ci_count=q["count"], lower=q["lower"], median=q["median"], upper=q["upper"],
                 ci_width=q["ci_width"])
    return st


def test_combine_posterior_one_rank_passes_quantiles_through():
    from sbd_b200.shard import ChainShard
    st = _with_quantiles(_samples(5, 3, 10, 12, seed=8), 2, 0.1)
    merged = ChainShard(3, 1, 0).combine_posterior(st)
    for m, d in zip(merged, st):
        assert set(m) == set(d)
        assert m["ci_alpha"] == 0.1 and m["ci_count"] == 15
        for k in ("lower", "median", "upper", "ci_width"):
            np.testing.assert_array_equal(m[k], d[k])


def _worker(rank, world, port, q, with_ci):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from sbd_b200.shard import ChainShard
    total = 4
    shard = ChainShard(total, world, rank)
    x = _samples(6, total, 13, 11, seed=9)[:, shard.chain_offset:shard.chain_offset + shard.n_local]
    mine = _with_quantiles(x, 2, 0.1) if (with_ci and rank == 1) else OP.stats(x, 2)
    try:
        merged = shard.combine_posterior(mine)
        q.put((rank, [sorted(d) for d in merged]))
    except ValueError as e:
        q.put((rank, str(e)))
    dist.destroy_process_group()


@pytest.mark.parametrize("with_ci", [True, False])
def test_two_gloo_ranks_refuse_quantiles(with_ci):
    """one rank with quantiles is enough: every rank raises, none waits in a collective"""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29100 + (os.getpid() % 300) + int(with_ci)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, with_ci)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    if with_ci:
        assert all(isinstance(m, str) and "one context" in m for _, m in res)
    else:
        assert all(isinstance(m, list) and "median" not in m[0] for _, m in res)


def test_signatures_and_python_refusals():
    import ctypes as C
    import sbd_b200
    from sbd_b200._lib import SIGNATURES
    res, args = SIGNATURES["sbd_set_posterior_quantiles"]
    assert res is C.c_int and args[1] is C.c_double
    res, args = SIGNATURES["sbd_posterior_quantiles"]
    assert res is C.c_int and len(args) == 7 and args[1] is C.c_int
    assert args[6]._type_ is C.c_longlong
    g = np.zeros((8, 8))
    for bad in (-0.1, 1.0, float("nan")):
        with pytest.raises(ValueError, match="post_ci"):
            sbd_b200.SAPG_algorithm_moffat(g, {"samples": 3}, post_levels=1, post_ci=bad)
