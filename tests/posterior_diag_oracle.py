"""Two-pass numpy restatement of the posterior diagnostics (DESIGN.md "Posterior statistics"; include/sbd.h
sbd_set_posterior_diagnostics / sbd_posterior_diagnostics) from a stack of samples, and their rank merge.  Test
infrastructure, built on oracle/posterior.py (block means, statistics, rank merge).

samples: [S, C, rows, cols] - S samples of each of C chains, already restricted to the accumulation window
ii = burnIn+1 .. samples."""
import numpy as np

from oracle.posterior import block_means, merge, stats


def auto_batch_len(n):
    """floor(sqrt(n)) (Flegal & Jones)"""
    return int(np.floor(np.sqrt(n))) if n > 0 else 0


def _triple(groups):
    """(mean, within, between) over the leading axis of per-group sample stacks groups[g] = [S, ...]; zeros for S = 0"""
    if groups[0].shape[0] == 0:
        z = np.zeros(groups[0].shape[1:])
        return z, z.copy(), z.copy()
    m = np.stack([g.mean(axis=0) for g in groups])
    within = sum(((g - mg[None]) ** 2).sum(axis=0) for g, mg in zip(groups, m))
    mean = m.mean(axis=0)
    between = ((m - mean[None]) ** 2).sum(axis=0)
    return mean, within, between


def diag_moments(var, batch_within, batch_between, half_within, half_between, n, C, b, B, h):
    """ESS, MCSE, Rhat_split from the sufficient statistics (batch means around the grand mean; split halves)."""
    nan = np.full(np.shape(var), np.nan)
    with np.errstate(divide="ignore", invalid="ignore"):
        if C * B >= 2:
            tau2 = b * (batch_within + B * batch_between) / (C * B - 1)
            ess, mcse = C * n * var / tau2, np.sqrt(tau2 / (C * n))
        else:
            ess, mcse = nan, nan
        if h >= 2:
            W = half_within / (2 * C * (h - 1))
            rhat = np.sqrt(((h - 1) / h * W + half_between / (2 * C - 1)) / W)
        else:
            rhat = nan
    return ess, mcse, rhat


def diagnostics(samples, levels, b=-1):
    """stats() extended, per block size, by the batch-means and split-half statistics: batch_len, n_batches, half_n,
    batch_mean, batch_within, batch_between, half_mean, half_within, half_between, ESS, MCSE, Rhat_split.
    b = -1: floor(sqrt(n)).  Batch q of chain c is the mean of samples q*b .. q*b+b-1; the first h = n//2 and the
    last h samples are the two halves, chain by chain in the order (c, half 1), (c, half 2)."""
    samples = np.asarray(samples, dtype=np.float64)
    S, C = samples.shape[:2]
    b = auto_batch_len(S) if b == -1 else int(b)
    B = S // b if b > 0 else 0
    h = S // 2
    out = stats(samples, levels)
    for j, d in enumerate(out):
        v = block_means(samples, 1 << j)                 # [S, C, bx, by]
        if B > 0:
            Y = v[:B * b].reshape((B, b) + v.shape[1:]).mean(axis=1)        # [B, C, bx, by]
            bm, bw, bb = _triple([Y[:, c] for c in range(C)])
        else:
            bm, bw, bb = _triple([np.zeros((0,) + v.shape[2:])])
        halves = []
        for c in range(C):
            halves += [v[:h, c], v[S - h:, c]]
        hm, hw, hb = _triple(halves)
        ess, mcse, rhat = diag_moments(d["var"], bw, bb, hw, hb, S, C, b, B, h)
        d.update(batch_len=b, n_batches=B, half_n=h, batch_mean=bm, batch_within=bw, batch_between=bb,
                 half_mean=hm, half_within=hw, half_between=hb, ESS=ess, MCSE=mcse, Rhat_split=rhat)
    return out


def merge_diagnostics(parts):
    """Rank merge of per-rank diagnostics (lists of (C_r, batch_mean_r, batch_within_r, batch_between_r, half_mean_r,
    half_within_r, half_between_r)), in rank order: batch statistics weighted by C_r, half statistics by 2 C_r."""
    _, bm, bw, bb = merge([(p[0], p[1], p[2], p[3]) for p in parts])
    _, hm, hw, hb = merge([(2 * p[0], p[4], p[5], p[6]) for p in parts])
    return bm, bw, bb, hm, hw, hb
