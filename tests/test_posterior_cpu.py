"""CPU tests of the posterior statistics (DESIGN.md "Posterior statistics"): oracle/posterior.py against direct numpy
with partial edge blocks, the rank merge against a single pass, R-hat for one chain, the host-side formulas of
host.posterior_moments, and ChainShard.combine_posterior over two gloo ranks."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

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


@pytest.mark.parametrize("shape,levels", [((243, 375), 7), ((7, 9), 7), ((64, 64), 4)])
def test_oracle_against_direct_numpy(shape, levels):
    S, C = 5, 3
    x = _samples(S, C, *shape, seed=1)
    st = OP.stats(x, levels)
    assert len(st) == levels
    for j, d in enumerate(st):
        s = 1 << j
        v = _loop_block_means(x, s)                                   # [S, C, bx, by]
        assert d["scale"] == s and d["n"] == S and d["chains"] == C
        assert d["mean"].shape == (-(-shape[0] // s), -(-shape[1] // s))
        np.testing.assert_allclose(d["mean"], v.mean(axis=(0, 1)), rtol=1e-13)
        # pooled variance = the sample variance of all C*n values
        flat = v.reshape(S * C, *v.shape[2:])
        np.testing.assert_allclose(d["var"], np.var(flat, axis=0, ddof=1), rtol=1e-12)
        np.testing.assert_allclose(d["std"], np.std(flat, axis=0, ddof=1), rtol=1e-12)
        # classic Gelman-Rubin from per-chain variances and the variance of the chain means
        Wd = np.var(v, axis=0, ddof=1).mean(axis=0)
        Bn = np.var(v.mean(axis=0), axis=0, ddof=1)
        R = np.sqrt(((S - 1) / S * Wd + Bn) / Wd)
        np.testing.assert_allclose(d["Rhat"], R, rtol=1e-12)


def test_partial_edge_blocks_divide_by_their_pixels():
    x = np.ones((1, 1, 7, 9))
    for j in range(4):
        np.testing.assert_array_equal(OP.block_means(x, 1 << j), np.ones((1, 1, -(-7 // (1 << j)), -(-9 // (1 << j)))))


def test_rank_merge_equals_single_pass():
    rng = np.random.default_rng(3)
    S, C = 6, 7
    x = _samples(S, C, 30, 21, seed=4)
    whole = OP.stats(x, 3)
    for trial in range(5):
        cuts = np.sort(rng.choice(np.arange(1, C), size=rng.integers(1, C - 1), replace=False))
        parts = np.split(np.arange(C), cuts)
        for j in range(3):
            per = [OP.stats(x[:, p], 3)[j] for p in parts]
            Cm, mean, within, between = OP.merge([(len(p), d["mean"], d["within"], d["between"])
                                                  for p, d in zip(parts, per)])
            assert Cm == C
            w = whole[j]
            for got, want in ((mean, w["mean"]), (within, w["within"]), (between, w["between"])):
                np.testing.assert_allclose(got, want, rtol=1e-13, atol=1e-13 * np.abs(want).max())


def test_rhat_is_nan_for_one_chain_or_one_sample():
    one = OP.stats(_samples(5, 1, 8, 8, seed=5), 2)
    assert all(np.all(np.isnan(d["Rhat"])) for d in one)
    assert np.all(np.isfinite(one[0]["var"]))
    single = OP.stats(_samples(1, 3, 8, 8, seed=6), 1)[0]
    assert np.all(np.isnan(single["Rhat"]))


def test_host_formulas_match_the_oracle():
    from sbd_b200.host import posterior_moments
    for S, C in ((5, 3), (4, 1), (1, 4), (2, 2)):
        d = OP.stats(_samples(S, C, 9, 11, seed=S * 10 + C), 1)[0]
        got = posterior_moments(d["mean"], d["within"], d["between"], S, C)
        want = OP.moments(d["mean"], d["within"], d["between"], S, C)
        for g, w in zip(got, want):
            np.testing.assert_allclose(g, w, rtol=1e-15, equal_nan=True)


def test_combine_posterior_one_rank_recomputes_the_moments():
    from sbd_b200.shard import ChainShard
    st = OP.stats(_samples(4, 3, 10, 12, seed=8), 2)
    merged = ChainShard(3, 1, 0).combine_posterior(st)
    for m, d in zip(merged, st):
        assert m["chains"] == 3 and m["n"] == 4 and m["scale"] == d["scale"]
        for k in ("mean", "within", "between", "var", "std", "Rhat"):
            np.testing.assert_allclose(m[k], d[k], rtol=1e-13)


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import posterior as OPw
    from sbd_b200.shard import ChainShard
    total = 4
    shard = ChainShard(total, world, rank)
    x = _samples(5, total, 37, 29, seed=9)
    mine = OPw.stats(x[:, shard.chain_offset:shard.chain_offset + shard.n_local], 4)
    merged = shard.combine_posterior(mine)
    q.put((rank, [{k: v for k, v in d.items()} for d in merged]))
    dist.destroy_process_group()


def test_two_gloo_ranks_combine_posterior():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29000 + (os.getpid() % 500)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = OP.stats(_samples(5, 4, 37, 29, seed=9), 4)
    for _, merged in res:
        for m, w in zip(merged, want):
            assert m["chains"] == 4 and m["n"] == 5
            for k in ("mean", "within", "between", "var", "std", "Rhat"):
                np.testing.assert_allclose(m[k], w[k], rtol=1e-12)
