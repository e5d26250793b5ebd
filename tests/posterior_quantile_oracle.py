"""numpy restatement of the posterior quantiles (DESIGN.md "Credible intervals and the median"; include/sbd.h
sbd_set_posterior_quantiles / sbd_posterior_quantiles): the device's block means in its own summation order and the
extended P^2 estimator, expression for expression.  Every operation below is one IEEE double operation (numpy
never contracts to FMA), and k_post_quantile evaluates the same expressions with __d*_rn, so the two agree bitwise.
Test infrastructure.

samples: [S, C, rows, cols] - S samples of each of C chains, already restricted to the accumulation window
ii = burnIn+1 .. samples."""
import numpy as np


def _pad_even(a):
    pr, pc = a.shape[-2] % 2, a.shape[-1] % 2
    return np.pad(a, [(0, 0)] * (a.ndim - 2) + [(0, pr), (0, pc)]) if pr or pc else a


def _nested_sum(a):
    """(top-left + bottom-left) + (top-right + bottom-right) over 2 x 2 groups, zeros outside"""
    a = _pad_even(a)
    return (a[..., 0::2, 0::2] + a[..., 1::2, 0::2]) + (a[..., 0::2, 1::2] + a[..., 1::2, 1::2])


def block_means_nested(x, s):
    """Block means at block size s = 2^j as k_post_blocks forms them: level 1 sums the pixels
    (v00 + v10) + (v01 + v11), every further level the four sums of the level below (tl + bl) + (tr + br), with zeros
    outside the image; then divides by the pixels the block holds."""
    x = np.asarray(x, dtype=np.float64)
    rows, cols = x.shape[-2:]
    v = x
    t = 1
    while t < s:
        v = _nested_sum(v)
        t *= 2
    bx, by = -(-rows // s), -(-cols // s)
    v = v[..., :bx, :by]
    ri = np.minimum((np.arange(bx) + 1) * s, rows) - np.arange(bx) * s
    ci = np.minimum((np.arange(by) + 1) * s, cols) - np.arange(by) * s
    return v / np.outer(ri, ci).astype(np.float64)


def marker_probs(alpha):
    """f_0 .. f_8, formed by exactly these double expressions (as sbd.cu forms them)"""
    a = float(alpha)
    return [0.0, a / 4, a / 2, 0.25 + a / 4, 0.5, 0.75 - a / 4, 1 - a / 2, 1 - a / 4, 1.0]


def _interp(v, N, p):
    """linear-interpolation quantile of the N sorted values v[0..N-1] (leading axis) at probability p"""
    h = float(N - 1) * p
    lo = int(np.floor(h))
    fr = h - np.floor(h)
    if fr == 0.0:
        return v[lo].copy()
    return v[lo] + fr * (v[lo + 1] - v[lo])


def p2(values, alpha):
    """Extended P^2 over a stream [S, C, ...] fed in (step, chain) order, one estimator per trailing element.
    Returns dict(lower, median, upper, count, q, n): q [9, ...] marker heights, n [9, ...] positions (N >= 9)."""
    values = np.asarray(values, dtype=np.float64)
    S, C = values.shape[:2]
    shape = values.shape[2:]
    stream = values.reshape((S * C,) + shape)
    N = S * C
    f = marker_probs(alpha)
    ps = (f[2], f[4], f[6])
    if N == 0:
        nan = np.full(shape, np.nan)
        return dict(lower=nan, median=nan.copy(), upper=nan.copy(), count=0, q=None, n=None)
    m = min(N, 9)
    q = np.sort(stream[:m], axis=0)                  # the insertion phase keeps the first values sorted
    if N < 9:
        lo, med, up = (_interp(q, N, p) for p in ps)
        return dict(lower=lo, median=med, upper=up, count=N, q=q, n=None)
    q = [q[i].copy() for i in range(9)]
    n = [np.full(shape, i + 1, dtype=np.int64) for i in range(9)]
    for t in range(9, N):
        x = stream[t]
        k = np.zeros(shape, dtype=np.int64)
        for i in range(1, 8):
            k = np.where(q[i] <= x, i, k)
        below = x < q[0]
        above = ~below & (x >= q[8])
        k = np.where(below, 0, np.where(above, 7, k))
        q[0] = np.where(below, x, q[0])
        q[8] = np.where(above, x, q[8])
        for i in range(1, 8):
            n[i] = n[i] + (i > k)
        n[8] = np.full(shape, t + 1, dtype=np.int64)   # the count after x
        for i in range(1, 8):
            d = (1.0 + float(t) * f[i]) - n[i].astype(np.float64)
            dr, dl = n[i + 1] - n[i], n[i] - n[i - 1]
            up = (d >= 1.0) & (dr > 1)
            mv = up | ((d <= -1.0) & (dl > 1))
            s = np.where(up, 1, -1)
            sd, ndr, ndl = s.astype(np.float64), dr.astype(np.float64), dl.astype(np.float64)
            dq1, dq0 = q[i + 1] - q[i], q[i] - q[i - 1]
            # parabolic: q_i + s/(dr+dl) [(dl+s) dq1/dr + (dr-s) dq0/dl] over the common denominator dr dl (dr+dl)
            num = ((ndl + sd) * ndl) * dq1 + ((ndr - sd) * ndr) * dq0
            den = (ndr * ndl) * (ndr + ndl)
            qp = q[i] + (sd * num) / den
            ql = q[i] + sd * np.where(s > 0, dq1 / ndr, dq0 / ndl)
            ok = (q[i - 1] < qp) & (qp < q[i + 1])
            q[i] = np.where(mv, np.where(ok, qp, ql), q[i])
            n[i] = np.where(mv, n[i] + s, n[i])
    return dict(lower=q[2].copy(), median=q[4].copy(), upper=q[6].copy(), count=N, q=np.stack(q), n=np.stack(n))


def quantiles(samples, levels, alpha):
    """One dict per block size 2^j, j < levels: lower, median, upper, count, ci_width - what the device returns for a
    run whose window samples are `samples`."""
    samples = np.asarray(samples, dtype=np.float64)
    out = []
    for j in range(levels):
        v = samples if j == 0 else block_means_nested(samples, 1 << j)
        r = p2(v, alpha)
        out.append(dict(lower=r["lower"], median=r["median"], upper=r["upper"], count=r["count"],
                        ci_width=r["upper"] - r["lower"]))
    return out
