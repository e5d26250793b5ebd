"""CPU tests of the posterior diagnostics (DESIGN.md "Posterior statistics"; include/sbd.h
sbd_set_posterior_diagnostics / sbd_posterior_diagnostics): tests/posterior_diag_oracle.py's batch means and split halves
against direct numpy with partial edge blocks, the rank merge against a single pass, the host formulas,
ChainShard.combine_posterior over two gloo ranks, statistical sanity on AR(1) and trending chains, and the refusal of
a batch length below -1."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import posterior_diag_oracle as PD  # noqa: E402
from oracle import posterior as OP  # noqa: E402


def _loop_block_means(x, s):
    """block means by explicit loops over the blocks of the last two axes"""
    rows, cols = x.shape[-2:]
    bx, by = -(-rows // s), -(-cols // s)
    out = np.zeros(x.shape[:-2] + (bx, by))
    for I in range(bx):
        for J in range(by):
            blk = x[..., I * s:min((I + 1) * s, rows), J * s:min((J + 1) * s, cols)]
            out[..., I, J] = blk.sum(axis=(-2, -1)) / (blk.shape[-2] * blk.shape[-1])
    return out


def _samples(S, C, rows, cols, seed):
    rng = np.random.default_rng(seed)
    chain_shift = rng.uniform(-1, 1, (1, C, 1, 1))
    return np.abs(100 + 20 * rng.standard_normal((S, C, rows, cols)) + 5 * chain_shift)


def _ar1(n, C, rho, seed, shape=(1, 1)):
    """C independent stationary AR(1) chains x_t = rho x_{t-1} + e_t, e ~ N(0, 1): marginal variance 1 / (1 - rho^2),
    asymptotic variance of the mean 1 / (1 - rho)^2"""
    rng = np.random.default_rng(seed)
    e = rng.standard_normal((n, C) + shape)
    x = np.empty_like(e)
    x[0] = e[0] / np.sqrt(1 - rho ** 2)
    for t in range(1, n):
        x[t] = rho * x[t - 1] + e[t]
    return x


# n a multiple of b, n not a multiple of b (B*b < n), odd n (middle sample dropped), automatic b, b > n
@pytest.mark.parametrize("S,b", [(12, 3), (14, 4), (13, -1), (9, 2), (16, -1), (5, 7)])
@pytest.mark.parametrize("shape,levels", [((37, 29), 4), ((7, 9), 4)])
def test_oracle_against_direct_numpy(S, b, shape, levels):
    C = 3
    x = _samples(S, C, *shape, seed=S * 7 + b)
    bb = int(np.floor(np.sqrt(S))) if b == -1 else b
    B, h = S // bb, S // 2
    st = PD.diagnostics(x, levels, b)
    for j, d in enumerate(st):
        v = _loop_block_means(x, 1 << j)                               # [S, C, bx, by]
        assert (d["batch_len"], d["n_batches"], d["half_n"]) == (bb, B, h)
        if B > 0:
            Y = np.stack([v[q * bb:(q + 1) * bb].mean(axis=0) for q in range(B)])     # [B, C, bx, by]
            np.testing.assert_allclose(d["batch_mean"], Y.mean(axis=(0, 1)), rtol=1e-13)
            # pooled batch means around the grand mean: within + B*between = sum over all C*B of (Y - grand mean)^2
            pooled = ((Y - Y.mean(axis=(0, 1))) ** 2).sum(axis=(0, 1))
            np.testing.assert_allclose(d["batch_within"] + B * d["batch_between"], pooled, rtol=1e-12)
            np.testing.assert_allclose(d["batch_between"], ((Y.mean(axis=0) - Y.mean(axis=(0, 1))) ** 2).sum(axis=0),
                                       rtol=1e-12)
            tau2 = bb * pooled / (C * B - 1) if C * B >= 2 else np.nan
            flat = v.reshape(S * C, *v.shape[2:])
            np.testing.assert_allclose(d["ESS"], C * S * np.var(flat, axis=0, ddof=1) / tau2, rtol=1e-12)
            np.testing.assert_allclose(d["MCSE"], np.sqrt(tau2 / (C * S)), rtol=1e-12)
        else:
            for k in ("batch_mean", "batch_within", "batch_between"):
                assert not np.any(d[k]) and d[k].shape == v.shape[2:]
            assert np.all(np.isnan(d["ESS"])) and np.all(np.isnan(d["MCSE"]))
        halves = np.stack([hv for c in range(C) for hv in (v[:h, c], v[S - h:, c])], axis=1)   # [h, 2C, bx, by]
        np.testing.assert_allclose(d["half_mean"], halves.mean(axis=(0, 1)), rtol=1e-13)
        Wd = np.var(halves, axis=0, ddof=1).mean(axis=0)
        Bn = np.var(halves.mean(axis=0), axis=0, ddof=1)
        np.testing.assert_allclose(d["half_within"], Wd * 2 * C * (h - 1), rtol=1e-12)
        np.testing.assert_allclose(d["Rhat_split"], np.sqrt(((h - 1) / h * Wd + Bn) / Wd), rtol=1e-12)
        if S % 2:                                                   # the middle sample takes no part in the halves
            y = x.copy()
            y[h] += 1e3
            d2 = PD.diagnostics(y, levels, b)[j]
            for k in ("half_mean", "half_within", "half_between"):
                np.testing.assert_array_equal(d2[k], d[k])


def test_rank_merge_equals_single_pass():
    rng = np.random.default_rng(3)
    S, C = 11, 7
    x = _samples(S, C, 30, 21, seed=4)
    whole = PD.diagnostics(x, 3, 3)
    keys = ("batch_mean", "batch_within", "batch_between", "half_mean", "half_within", "half_between")
    for trial in range(5):
        cuts = np.sort(rng.choice(np.arange(1, C), size=rng.integers(1, C - 1), replace=False))
        parts = np.split(np.arange(C), cuts)
        for j in range(3):
            per = [PD.diagnostics(x[:, p], 3, 3)[j] for p in parts]
            got = PD.merge_diagnostics([(len(p),) + tuple(d[k] for k in keys) for p, d in zip(parts, per)])
            for g, k in zip(got, keys):
                want = whole[j][k]
                np.testing.assert_allclose(g, want, rtol=1e-13, atol=1e-13 * np.abs(want).max())


def test_host_formulas_match_the_oracle():
    from sbd_b200.host import posterior_diagnostics
    for S, C, b in ((9, 3, 2), (16, 1, -1), (5, 2, 7), (1, 4, -1), (3, 1, 1)):
        d = PD.diagnostics(_samples(S, C, 9, 11, seed=S * 10 + C), 1, b)[0]
        got = posterior_diagnostics(d["var"], d["batch_within"], d["batch_between"], d["half_within"],
                                    d["half_between"], S, C, d["batch_len"], d["n_batches"], d["half_n"])
        for g, k in zip(got, ("ESS", "MCSE", "Rhat_split")):
            np.testing.assert_allclose(g, d[k], rtol=1e-15, equal_nan=True)


@pytest.mark.parametrize("rho", [0.0, 0.5, 0.9])
def test_batch_means_variance_on_ar1_chains(rho):
    n, C = 40000, 4
    d = PD.diagnostics(_ar1(n, C, rho, seed=int(rho * 10) + 1), 1)[0]
    b, B = d["batch_len"], d["n_batches"]
    assert b == 200 and B == 200
    tau2 = d["MCSE"][0, 0] ** 2 * C * n
    want = (1 / (1 - rho ** 2)) * (1 + rho) / (1 - rho)
    assert abs(tau2 / want - 1) < 0.2, (rho, tau2 / want)
    # ESS = C n var / tau2: about C n (1 - rho) / (1 + rho)
    assert abs(d["ESS"][0, 0] / (C * n * (1 - rho) / (1 + rho)) - 1) < 0.25
    assert d["Rhat_split"][0, 0] < 1.01                     # stationary chains


def test_split_rhat_sees_a_trend_in_one_chain():
    n = 2000
    rng = np.random.default_rng(11)
    x = (rng.standard_normal(n) + 3.0 * np.arange(n) / n)[:, None, None, None]    # one chain
    d = PD.diagnostics(x, 1)[0]
    assert np.isnan(d["Rhat"][0, 0])                         # classic Rhat needs two chains
    assert d["Rhat_split"][0, 0] > 1.2
    still = PD.diagnostics(_ar1(n, 1, 0.3, seed=12), 1)[0]
    assert still["Rhat_split"][0, 0] < 1.05


def test_combine_posterior_one_rank():
    """with diagnostics: merged statistics recomputed; without: exactly the fields and values of the statistics"""
    from sbd_b200.shard import ChainShard
    x = _samples(9, 3, 10, 12, seed=8)
    plain = OP.stats(x, 2)
    merged = ChainShard(3, 1, 0).combine_posterior(plain)
    for m, d in zip(merged, plain):
        assert set(m) == set(d)
    st = PD.diagnostics(x, 2, 2)
    merged = ChainShard(3, 1, 0).combine_posterior(st)
    for m, d in zip(merged, st):
        assert set(m) == set(d)
        assert (m["batch_len"], m["n_batches"], m["half_n"]) == (2, 4, 4)
        for k in ("batch_mean", "batch_within", "batch_between", "half_mean", "half_within", "half_between", "ESS",
                  "MCSE", "Rhat_split"):
            np.testing.assert_allclose(m[k], d[k], rtol=1e-13)


def _worker(rank, world, port, q, b):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import posterior_diag_oracle as PDw
    from sbd_b200.shard import ChainShard
    total = 4
    shard = ChainShard(total, world, rank)
    x = _samples(13, total, 37, 29, seed=9)
    mine = PDw.diagnostics(x[:, shard.chain_offset:shard.chain_offset + shard.n_local], 4, b)
    if b == 3 and rank == 1:                    # a rank that batched differently is refused
        for d in mine:
            d["batch_len"], d["n_batches"] = 4, 3
    try:
        merged = shard.combine_posterior(mine)
        q.put((rank, [{k: v for k, v in d.items()} for d in merged]))
    except ValueError as e:
        q.put((rank, str(e)))
    dist.destroy_process_group()


@pytest.mark.parametrize("b", [-1, 3])
def test_two_gloo_ranks_combine_posterior(b):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 400) + (b + 1)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, b)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    if b == 3:
        assert all(isinstance(m, str) and "batch_len" in m for _, m in res)
        return
    want = PD.diagnostics(_samples(13, 4, 37, 29, seed=9), 4, b)
    for _, merged in res:
        for m, w in zip(merged, want):
            assert m["chains"] == 4 and m["n"] == 13 and (m["batch_len"], m["n_batches"], m["half_n"]) == (3, 4, 6)
            for k in ("mean", "within", "between", "var", "batch_mean", "batch_within", "batch_between", "half_mean",
                      "half_within", "half_between", "ESS", "MCSE", "Rhat_split"):
                np.testing.assert_allclose(m[k], w[k], rtol=1e-12)


def test_batch_len_below_minus_one_is_refused():
    """before the library is reached (the Python mirror), and by the C entry point's declared prototype"""
    import sbd_b200
    from sbd_b200._lib import SIGNATURES
    g = np.zeros((8, 8))
    for f, args in ((sbd_b200.SAPG_algorithm_Guassian, (g, {"samples": 3}, {})),
                    (sbd_b200.SAPG_algorithm_moffat, (g, {"samples": 3})),
                    (sbd_b200.SAPG_algorithm_laplace, (g, {"samples": 3, "x": g}))):
        with pytest.raises(ValueError, match="post_batch"):
            f(*args, post_levels=1, post_batch=-2)
    assert SIGNATURES["sbd_set_posterior_diagnostics"][1][1].__name__ == "c_int"
    assert len(SIGNATURES["sbd_posterior_diagnostics"][1]) == 11
