"""Two-pass numpy restatement of the posterior statistics (DESIGN.md "Posterior statistics"; include/sbd.h
sbd_set_posterior / sbd_posterior_stats) from a stack of samples, and the rank merge.  Test infrastructure.

samples: [S, C, rows, cols] - S samples of each of C chains, already restricted to the accumulation window
ii = burnIn+1 .. samples."""
import numpy as np


def block_means(x, s):
    """Block means of the last two axes at block size s; partial edge blocks divide by the pixels they hold."""
    x = np.asarray(x, dtype=np.float64)
    rows, cols = x.shape[-2:]
    bx, by = -(-rows // s), -(-cols // s)
    pr, pc = bx * s - rows, by * s - cols
    pad = [(0, 0)] * (x.ndim - 2) + [(0, pr), (0, pc)]
    xs = np.pad(x, pad).reshape(x.shape[:-2] + (bx, s, by, s)).sum(axis=(-3, -1))
    ri = np.minimum((np.arange(bx) + 1) * s, rows) - np.arange(bx) * s
    ci = np.minimum((np.arange(by) + 1) * s, cols) - np.arange(by) * s
    return xs / np.outer(ri, ci)


def moments(mean, within, between, n, C):
    """var, std, Rhat from the sufficient statistics (classic Gelman-Rubin, not split, not rank-normalised)."""
    nan = np.full(np.shape(within), np.nan)
    with np.errstate(divide="ignore", invalid="ignore"):
        var = (within + n * between) / (C * n - 1) if C * n >= 2 else nan
        if C >= 2 and n >= 2:
            W = within / (C * (n - 1))
            rhat = np.sqrt(((n - 1) / n * W + between / (C - 1)) / W)
        else:
            rhat = nan
    return var, np.sqrt(var), rhat


def stats(samples, levels):
    """One dict per block size 2^j, j < levels: scale, n, chains, mean, within, between, var, std, Rhat."""
    samples = np.asarray(samples, dtype=np.float64)
    S, C = samples.shape[:2]
    out = []
    for j in range(levels):
        v = block_means(samples, 1 << j)                 # [S, C, bx, by]
        if S == 0:
            z = np.zeros(v.shape[2:])
            m_c = np.zeros((C,) + z.shape)
            mean, within, between = z, z.copy(), z.copy()
        else:
            m_c = v.mean(axis=0)                          # per-chain mean
            within = ((v - m_c[None]) ** 2).sum(axis=(0, 1))
            mean = m_c.mean(axis=0)
            between = ((m_c - mean[None]) ** 2).sum(axis=0)
        var, std, rhat = moments(mean, within, between, S, C)
        out.append(dict(scale=1 << j, n=S, chains=C, mean=mean, within=within, between=between, var=var, std=std,
                        Rhat=rhat))
    return out


def merge(parts):
    """Rank merge of per-rank statistics (lists of (C_r, mean_r, within_r, between_r)), in rank order."""
    C = sum(p[0] for p in parts)
    mean = sum(p[0] * p[1] for p in parts) / C
    within = sum(p[2] for p in parts)
    between = sum(p[3] + p[0] * (p[1] - mean) ** 2 for p in parts)
    return C, mean, within, between
