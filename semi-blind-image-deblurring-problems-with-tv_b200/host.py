"""Host-side mirror of the reference's MATLAB interface for the hot path.

Same names, argument meaning and error behaviour as the .m files they stand in
for (cited per function); every one of them forwards to the CUDA engine through
the C ABI (`_lib.py`).  Arrays follow numpy's `a[i, j]` == MATLAB `a(i+1, j+1)`;
they are handed to the library in MATLAB (column-major) memory order.
"""
import ctypes as C

import numpy as np

from ._lib import lib, sbd_params, sbd_traces, SbdError, c_double_p, SBD_N_PHASES, SBD_N_GEOM

GAUSSIAN, MOFFAT, LAPLACE = 0, 1, 2
K_PSF, K_DPSI0, K_DPSI1 = 0, 1, 2
OP_A, OP_AT, OP_D0, OP_D1 = 0, 1, 2, 3


def _f(a):
    """float64, column-major (MATLAB layout), owning a contiguous buffer."""
    return np.asfortranarray(np.asarray(a, dtype=np.float64))


def _p(a):
    return a.ctypes.data_as(c_double_p) if a is not None else None


def _psi(psi):
    v = np.zeros(2)
    psi = np.atleast_1d(np.asarray(psi, dtype=np.float64))
    v[:psi.size] = psi[:2]
    return v


def posterior_moments(mean, within, between, n, chains):
    """var, std and Gelman-Rubin Rhat from the sufficient statistics sbd_posterior_stats returns (DESIGN.md
    "Posterior statistics"): n samples per chain, `chains` chains.
      var  = (within + n*between) / (C*n - 1)                     (NaN for C*n < 2)
      W    = within / (C(n-1)),  B/n = between / (C-1),  V = (n-1)/n * W + B/n,  Rhat = sqrt(V / W)
                                                                  (NaN for C < 2 or n < 2)"""
    within = np.asarray(within, dtype=np.float64)
    between = np.asarray(between, dtype=np.float64)
    n, C_ = int(n), int(chains)
    nan = np.full(within.shape, np.nan)
    with np.errstate(divide="ignore", invalid="ignore"):
        var = (within + n * between) / (C_ * n - 1) if C_ * n >= 2 else nan.copy()
        if C_ >= 2 and n >= 2:
            W = within / (C_ * (n - 1))
            V = (n - 1) / n * W + between / (C_ - 1)
            rhat = np.sqrt(V / W)
        else:
            rhat = nan.copy()
    return var, np.sqrt(var), rhat


def posterior_diagnostics(var, batch_within, batch_between, half_within, half_between, n, chains, batch_len,
                          n_batches, half_n):
    """ESS, MCSE and split-Rhat from the sufficient statistics sbd_posterior_diagnostics returns and var of
    posterior_moments (DESIGN.md "Posterior statistics"): n samples per chain, `chains` chains, batch length b,
    B = n_batches batches, half length h = half_n.
      tau2 = b (batch_within + B batch_between) / (C B - 1)                (NaN for C B < 2)
      ESS  = C n var / tau2,  MCSE = sqrt(tau2 / (C n))
      W    = half_within / (2C(h-1)),  Bh = half_between / (2C-1),  Rhat_split = sqrt(((h-1)/h W + Bh) / W)
                                                                          (NaN for h < 2)"""
    var = np.asarray(var, dtype=np.float64)
    n, C_, b, B, h = int(n), int(chains), int(batch_len), int(n_batches), int(half_n)
    nan = np.full(var.shape, np.nan)
    with np.errstate(divide="ignore", invalid="ignore"):
        if C_ * B >= 2:
            tau2 = b * (np.asarray(batch_within, dtype=np.float64) + B * np.asarray(batch_between, dtype=np.float64)) \
                / (C_ * B - 1)
            ess, mcse = C_ * n * var / tau2, np.sqrt(tau2 / (C_ * n))
        else:
            ess, mcse = nan.copy(), nan.copy()
        if h >= 2:
            W = np.asarray(half_within, dtype=np.float64) / (2 * C_ * (h - 1))
            Bh = np.asarray(half_between, dtype=np.float64) / (2 * C_ - 1)
            rhat = np.sqrt(((h - 1) / h * W + Bh) / W)
        else:
            rhat = nan.copy()
    return ess, mcse, rhat


class Engine:
    """One libsbd context: fixed image size, PSF family and GPU."""

    def __init__(self, rows, cols, psf_size=7, model=GAUSSIAN, phi=0.0, max_batch=1, device=0):
        self.rows, self.cols, self.psf_size = int(rows), int(cols), int(psf_size)
        self.model, self.phi, self.max_batch, self.device = int(model), float(phi), int(max_batch), int(device)
        self._h = C.c_void_p()
        rc = lib.sbd_create(C.byref(self._h), self.rows, self.cols, self.psf_size, self.model,
                            self.phi, self.max_batch, self.device)
        if rc != 0:
            raise SbdError(rc, lib.sbd_last_error(None).decode())

    # -- plumbing ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib.sbd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise SbdError(rc, lib.sbd_last_error(self._h).decode())

    def _img(self, x, name="x"):
        x = np.asarray(x, dtype=np.float64)
        if x.ndim == 2:
            x = x[None]
        if x.ndim != 3 or x.shape[1:] != (self.rows, self.cols):
            raise ValueError(f"{name}: expected [batch,]{self.rows}x{self.cols}, got {x.shape}")
        if x.shape[0] > self.max_batch:
            raise ValueError(f"{name}: batch {x.shape[0]} exceeds max_batch {self.max_batch}")
        # [b, i, j] -> memory order b, j, i  (each image column-major)
        return np.ascontiguousarray(x.transpose(0, 2, 1)), x.shape[0]

    def _unimg(self, buf, batch, squeeze):
        out = buf.reshape(batch, self.cols, self.rows).transpose(0, 2, 1)
        return np.ascontiguousarray(out[0]) if squeeze else np.ascontiguousarray(out)

    @property
    def launches(self):
        return int(lib.sbd_launch_count(self._h))

    def synchronize(self):
        self._check(lib.sbd_synchronize(self._h))

    def set_profile(self, on=True):
        self._check(lib.sbd_set_profile(self._h, int(bool(on))))

    def set_option(self, name, value):
        """Launch-geometry override (include/sbd.h: sbd_set_option); -1 restores the automatic choice."""
        self._check(lib.sbd_set_option(self._h, name.encode(), int(value)))

    def geometry(self, batch=1):
        """dict of the launch geometry libsbd would use for a batch of `batch` images."""
        out = (C.c_int * SBD_N_GEOM)()
        self._check(lib.sbd_get_geometry(self._h, int(batch), out))
        keys = ("levels", "chamb_seg", "chamb_grid_x", "chamb_grid_y", "tv_seg", "tv_grid_x", "tv_grid_y", "rows_line_pairs",
                "coop_blocks_per_image", "coop_units_per_warp")
        return dict(zip(keys, list(out)))

    def phase_times(self):
        """{phase: (milliseconds, event pairs)} of the last run's main loop."""
        ms = (C.c_double * SBD_N_PHASES)()
        calls = (C.c_longlong * SBD_N_PHASES)()
        self._check(lib.sbd_phase_times(self._h, ms, calls))
        return {lib.sbd_phase_name(i).decode(): (ms[i], int(calls[i])) for i in range(SBD_N_PHASES)}

    # -- PSF --------------------------------------------------------------
    def psf_taps(self, psi, which=K_PSF):
        t = self.psf_size
        out = np.zeros(t * t)
        self._check(lib.sbd_psf_taps(self._h, _p(_psi(psi)), which, _p(out)))
        return out.reshape(t, t).T.copy()

    def psf_spectrum(self, psi, which=K_PSF):
        n = self.rows * self.cols
        re, im = np.zeros(n), np.zeros(n)
        self._check(lib.sbd_psf_spectrum(self._h, _p(_psi(psi)), which, _p(re), _p(im)))
        return (re + 1j * im).reshape(self.cols, self.rows).T.copy()

    # -- operators ----------------------------------------------------------
    def blur(self, x, psi, op=OP_A):
        squeeze = np.asarray(x).ndim == 2
        buf, b = self._img(x)
        out = np.empty_like(buf)
        self._check(lib.sbd_blur(self._h, _p(buf), _p(_psi(psi)), op, _p(out), b))
        return self._unimg(out, b, squeeze)

    def tvnorm(self, x):
        squeeze = np.asarray(x).ndim == 2
        buf, b = self._img(x)
        out = np.zeros(b)
        self._check(lib.sbd_tvnorm(self._h, _p(buf), _p(out), b))
        return float(out[0]) if squeeze else out

    def diff(self, x, axis):
        squeeze = np.asarray(x).ndim == 2
        buf, b = self._img(x)
        out = np.empty_like(buf)
        self._check(lib.sbd_diff(self._h, _p(buf), axis, _p(out), b))
        return self._unimg(out, b, squeeze)

    def tvprox(self, g, lam, maxiter, tol=1e-3, tau=0.249, dualvars=None):
        """-> f, px, py, iters, err (per image)."""
        squeeze = np.asarray(g).ndim == 2
        buf, b = self._img(g, "g")
        f = np.empty_like(buf); px = np.empty_like(buf); py = np.empty_like(buf)
        iters = (C.c_int * b)(); err = np.zeros(b)
        dpx = dpy = None
        if dualvars is not None:
            dpx, _ = self._img(dualvars[0], "px")
            dpy, _ = self._img(dualvars[1], "py")
        self._check(lib.sbd_tvprox(self._h, _p(buf), float(lam), int(maxiter), float(tol), float(tau),
                                   _p(dpx), _p(dpy), _p(f), _p(px), _p(py), iters, _p(err), b))
        it = np.array(list(iters))
        if squeeze:
            return (self._unimg(f, b, True), self._unimg(px, b, True), self._unimg(py, b, True), int(it[0]), float(err[0]))
        return self._unimg(f, b, False), self._unimg(px, b, False), self._unimg(py, b, False), it, err

    def likelihood(self, x, y, psi, sigma2, theta=0.0, want_grad=True):
        """-> dict(f, grad_psi0, grad_psi1, gradF_sigma, g, logPi[, gradF])."""
        xb, _ = self._img(x); yb, _ = self._img(y, "y")
        scal = np.zeros(6)
        gf = np.empty_like(xb) if want_grad else None
        self._check(lib.sbd_likelihood(self._h, _p(xb), _p(yb), _p(_psi(psi)), float(sigma2), float(theta),
                                       _p(scal), _p(gf)))
        out = dict(f=scal[0], grad_psi0=scal[1], grad_psi1=scal[2], gradF_sigma=scal[3], g=scal[4], logPi=scal[5])
        if want_grad:
            out["gradF"] = self._unimg(gf, 1, True)
        return out

    # -- setup stage of the demos ---------------------------------------------
    def max_eigenval(self, psi, tol=1e-4, max_iter=10000, x0=None, seed=1):
        """utils/max_eigenval_Gaussian_Moffat.m / max_eigenval_Laplace.m -> (val, iterations)."""
        x0b = self._img(x0, "x0")[0] if x0 is not None else None
        val = C.c_double(); it = C.c_int()
        self._check(lib.sbd_max_eigenval(self._h, _p(_psi(psi)), _p(x0b), float(tol), int(max_iter), int(seed),
                                         C.byref(val), C.byref(it)))
        return val.value, it.value

    def observe(self, x, psi, bsnr, noise=None, seed=1):
        """run_Gaussian_demo.m:145-168 -> (y, sigma, ||Ax - mean(Ax)||_F)."""
        xb, _ = self._img(x)
        nb = self._img(noise, "noise")[0] if noise is not None else None
        y = np.empty_like(xb); sg = C.c_double(); nr = C.c_double()
        self._check(lib.sbd_observe(self._h, _p(xb), _p(_psi(psi)), float(bsnr), _p(nb), int(seed), _p(y),
                                    C.byref(sg), C.byref(nr)))
        return self._unimg(y, 1, True), sg.value, nr.value

    # -- post-SAPG MAP estimate -----------------------------------------------
    def salsa_tv(self, y, psi, tau, mu, maxiter=500, tolA=1e-5, tv_iters=10, x_true=None):
        """SALSA_v2 as the demos call it (run_Gaussian_demo.m:229-242) ->
        dict(x, objective, distance, mses, n_outer, numA, numAt)."""
        yb, _ = self._img(y, "y")
        xt = self._img(x_true, "x_true")[0] if x_true is not None else None
        x = np.empty_like(yb)
        obj = np.zeros(maxiter + 1); dist = np.zeros(maxiter); mses = np.zeros(maxiter + 1)
        n = C.c_int()
        self._check(lib.sbd_salsa_tv(self._h, _p(yb), _p(_psi(psi)), float(tau), float(mu), int(maxiter), float(tolA),
                                     int(tv_iters), _p(xt), _p(x), _p(obj), _p(dist), _p(mses), C.byref(n)))
        k = n.value
        return dict(x=self._unimg(x, 1, True), objective=obj[:k + 1], distance=dist[:k],
                    mses=mses[:k + 1] if x_true is not None else np.zeros(0), n_outer=k, numA=k + 1, numAt=1)

    # -- SAPG -----------------------------------------------------------------
    def set_posterior(self, levels):
        """sbd_set_posterior: 0 off, L in 1..7 accumulates posterior moments at block sizes 1 .. 2^(L-1) in every
        following run (sticky on the context)."""
        self._check(lib.sbd_set_posterior(self._h, int(levels)))

    def posterior_stats(self, level):
        """Statistics of the last run at block size 2^level: dict(scale, n, chains, mean, within, between, var, std,
        Rhat), images ceil(rows/s) x ceil(cols/s)."""
        s = 1 << int(level)
        bx, by = -(-self.rows // s), -(-self.cols // s)
        bufs = [np.zeros(bx * by) for _ in range(3)]
        n, ch = C.c_int(), C.c_int()
        self._check(lib.sbd_posterior_stats(self._h, int(level), *[_p(b) for b in bufs], C.byref(n), C.byref(ch)))
        mean, within, between = (b.reshape(by, bx).T.copy() for b in bufs)
        var, std, rhat = posterior_moments(mean, within, between, n.value, ch.value)
        return dict(scale=s, n=n.value, chains=ch.value, mean=mean, within=within, between=between, var=var, std=std,
                    Rhat=rhat)

    def set_posterior_diagnostics(self, batch_len):
        """sbd_set_posterior_diagnostics: 0 off, -1 batch length floor(sqrt(n)), b >= 1 batch length b; every
        following run with posterior statistics also accumulates batch means and split halves (sticky)."""
        self._check(lib.sbd_set_posterior_diagnostics(self._h, int(batch_len)))

    def posterior_diagnostics(self, level, stats=None):
        """Diagnostics of the last run at block size 2^level: dict(batch_mean, batch_within, batch_between, half_mean,
        half_within, half_between, batch_len, n_batches, half_n, ESS, MCSE, Rhat_split), images ceil(rows/s) x
        ceil(cols/s).  ESS and MCSE use var of `stats` (posterior_stats(level) of the same run, read if not given)."""
        s = 1 << int(level)
        bx, by = -(-self.rows // s), -(-self.cols // s)
        bufs = [np.zeros(bx * by) for _ in range(6)]
        b, nb, h = C.c_int(), C.c_int(), C.c_int()
        self._check(lib.sbd_posterior_diagnostics(self._h, int(level), *[_p(q) for q in bufs], C.byref(b),
                                                  C.byref(nb), C.byref(h)))
        names = ("batch_mean", "batch_within", "batch_between", "half_mean", "half_within", "half_between")
        d = {k: q.reshape(by, bx).T.copy() for k, q in zip(names, bufs)}
        d.update(batch_len=b.value, n_batches=nb.value, half_n=h.value)
        st = self.posterior_stats(level) if stats is None else stats
        d["ESS"], d["MCSE"], d["Rhat_split"] = posterior_diagnostics(
            st["var"], d["batch_within"], d["batch_between"], d["half_within"], d["half_between"], st["n"],
            st["chains"], b.value, nb.value, h.value)
        return d

    def sapg(self, y, prm, X0=None, x_true=None, noise=None, want_X_warm=True, want_X_mean=False, post_levels=0,
             post_batch=0):
        """Run sbd_sapg_run.  `prm` is a filled sbd_params; noise (optional)
        is [(warmup-1)+(samples-1), n_chains, rows, cols].  post_levels L > 0 adds out["posterior"]: one
        `posterior_stats` dict per block size 1 .. 2^(L-1); post_batch (-1: floor(sqrt(n)), b >= 1; needs L > 0)
        adds the `posterior_diagnostics` fields to each.  The context is left with both off."""
        yb, _ = self._img(y, "y")
        x0b = self._img(X0, "X0")[0] if X0 is not None else None
        xtb = self._img(x_true, "x_true")[0] if x_true is not None else None
        nb = None
        if noise is not None:
            noise = np.asarray(noise, dtype=np.float64)
            draws = max(prm.warmup - 1, 0) + max(prm.samples - 1, 0)
            if noise.shape != (draws, prm.n_chains, self.rows, self.cols):
                raise ValueError(f"noise: expected {(draws, prm.n_chains, self.rows, self.cols)}, got {noise.shape}")
            nb = np.ascontiguousarray(noise.transpose(0, 1, 3, 2))
        S, W, nch = prm.samples, prm.warmup, prm.n_chains
        nm = max(S - prm.burnIn, 0)
        tr = sbd_traces()
        bufs = {}
        for name in ("thetas", "sigmas", "psi0", "psi1", "grad_theta", "grad_psi0", "grad_psi1", "grad_sigma",
                     "logPiTraceX", "gXTrace", "err_psf", "err_sample", "tol_theta", "tol_psi0", "tol_psi1", "tol_sigma"):
            bufs[name] = np.zeros(S)
        bufs["logPiTrace_WU"] = np.zeros(max(W, 1))
        for name in ("mean_theta", "mean_psi0", "mean_psi1", "mean_sigma"):
            bufs[name] = np.zeros(max(nm, 1))
        for name, b in bufs.items():
            setattr(tr, name, _p(b))
        ck = np.zeros(S, dtype=np.int32)
        tr.chambolle_iters = ck.ctypes.data_as(C.POINTER(C.c_int32))
        xl = np.zeros(nch * self.rows * self.cols)
        tr.X_last = _p(xl)
        xw = xm = None
        if want_X_warm:
            xw = np.zeros(nch * self.rows * self.cols); tr.X_warm = _p(xw)
        if want_X_mean:
            xm = np.zeros(self.rows * self.cols); tr.X_mean = _p(xm)
        self.set_posterior(post_levels)
        try:
            self.set_posterior_diagnostics(post_batch)
            self._check(lib.sbd_sapg_run(self._h, _p(yb), _p(x0b), _p(xtb), C.byref(prm), _p(nb), C.byref(tr)))
            posterior = [self.posterior_stats(j) for j in range(int(post_levels))]
            if post_batch:
                for j, st in enumerate(posterior):
                    st.update(self.posterior_diagnostics(j, st))
        finally:
            if post_levels:
                lib.sbd_set_posterior(self._h, 0)
            if post_batch:
                lib.sbd_set_posterior_diagnostics(self._h, 0)
        out = dict(bufs)
        if post_levels:
            out["posterior"] = posterior
        out["logPiTrace_WU"] = bufs["logPiTrace_WU"][:W]
        for name in ("mean_theta", "mean_psi0", "mean_psi1", "mean_sigma"):
            out[name] = bufs[name][:nm]
        out["chambolle_iters"] = ck
        out["X_last"] = self._unimg(xl, nch, False)
        if xw is not None:
            out["X_warm"] = self._unimg(xw, nch, False)
        if xm is not None:
            out["X_mean"] = self._unimg(xm, 1, True)
        out["EB"] = np.array(list(tr.EB))
        out["err_warm0"] = tr.err_warm0
        out["seconds"] = tr.seconds
        out["seconds_main"] = tr.seconds_main
        out["launches_main"] = int(tr.launches_main)
        out["last_samp"] = tr.last_samp
        return out


_engines = {}


def engine_for(shape, psf_size=7, model=GAUSSIAN, phi=0.0, max_batch=1, device=0):
    """Cached context per (size, PSF family, device) - the analogue of the
    persistent context a MEX file keeps behind mexLock."""
    key = (int(shape[0]), int(shape[1]), int(psf_size), int(model), float(phi), int(device))
    e = _engines.get(key)
    if e is None or e.max_batch < max_batch or e._h is None:
        if e is not None:
            e.close()
        e = Engine(shape[0], shape[1], psf_size, model, phi, max_batch, device)
        _engines[key] = e
    return e


# ---------------------------------------------------------------------------
# utils/*.m mirrors
# ---------------------------------------------------------------------------
def _taps(model, t, psi, phi, which):
    return engine_for((max(t, 16), max(t, 16)), t, model, phi).psf_taps(psi, which)


def Gaussian_psf(taille, w1, w2, phi):
    """utils/Gaussian_psf.m:2-19."""
    return _taps(GAUSSIAN, taille, (w1, w2), phi, K_PSF)


psf_gaussian = Gaussian_psf             # utils/psf_gaussian.m:2-19


def psf_moffat(size, a, b):
    """utils/psf_moffat.m:2-20."""
    return _taps(MOFFAT, size, (a, b), 0.0, K_PSF)


def psf_laplace(size, b):
    """utils/psf_laplace.m:1-13."""
    return _taps(LAPLACE, size, (b,), 0.0, K_PSF)


def gaussian_fft(im_size, taille, w1, w2, phi):
    """resize(Gaussian_psf(taille,w1,w2,phi), im_size) - run_Gaussian_demo.m:128."""
    return engine_for(im_size, taille, GAUSSIAN, phi).psf_spectrum((w1, w2), K_PSF)


def diff_fftgaus_w1(im_size, taille, w1, w2, phi):
    """utils/diff_fftgaus_w1.m:2-26."""
    return engine_for(im_size, taille, GAUSSIAN, phi).psf_spectrum((w1, w2), K_DPSI0)


def diff_fftgaus_w2(im_size, taille, w1, w2, phi):
    """utils/diff_fftgaus_w2.m:2-26."""
    return engine_for(im_size, taille, GAUSSIAN, phi).psf_spectrum((w1, w2), K_DPSI1)


def moffat_psf(im_shape, size, a, b):
    """utils/moffat_psf.m:2-23."""
    return engine_for(im_shape, size, MOFFAT).psf_spectrum((a, b), K_PSF)


def diff_moffat_alpha(im_shape, size, a, b):
    """utils/diff_moffat_alpha.m:1-22."""
    return engine_for(im_shape, size, MOFFAT).psf_spectrum((a, b), K_DPSI0)


def diff_moffat_beta(im_shape, size, a, b):
    """utils/diff_moffat_beta.m:1-23."""
    return engine_for(im_shape, size, MOFFAT).psf_spectrum((a, b), K_DPSI1)


def laplace_psf(im_shape, size, b):
    """utils/laplace_psf.m:1-15."""
    return engine_for(im_shape, size, LAPLACE).psf_spectrum((b,), K_PSF)


def diff_laplace_b(im_shape, size, b):
    """utils/diff_laplace_b.m:1-19."""
    return engine_for(im_shape, size, LAPLACE).psf_spectrum((b,), K_DPSI0)


def _tv_engine(shape):
    """TV entry points accept any size >= 2 (no FFT involved): psf_size 1."""
    return engine_for(shape, 1, GAUSSIAN, 0.0)


def TVnorm(x):
    """utils/TVnorm.m:1-2."""
    x = np.asarray(x)
    return _tv_engine(x.shape).tvnorm(x)


def diffh(x):
    """SALSA/diffh.m:1-3."""
    x = np.asarray(x)
    return _tv_engine(x.shape).diff(x, 1)


def diffv(x):
    """SALSA/diffv.m:1-3."""
    x = np.asarray(x)
    return _tv_engine(x.shape).diff(x, 0)


def chambolle_prox_TV_stop(g, *varargin):
    """[f, px, py] = chambolle_prox_TV_stop(g, 'lambda', l, 'maxiter', K, ...)
    utils/chambolle_prox_TV_stop.m:1-150: same option names (case-insensitive,
    :88), same defaults (:77-81), 'dualvars' = [px py] (:99-107, square only)
    and the same failure when 'maxiter' is omitted (:80,:131)."""
    g = np.asarray(g, dtype=np.float64)
    if len(varargin) % 2 != 0:
        raise ValueError("Wrong number of required parameters")            # :60-62
    tau, tol, lam, maxiter, dual = 0.249, 1e-3, 1.0, None, None
    for i in range(0, len(varargin) - 1, 2):
        name = str(varargin[i]).upper(); val = varargin[i + 1]
        if name == "LAMBDA":
            lam = float(val)
        elif name == "VERBOSE":
            pass
        elif name == "TOL":
            tol = float(val)
        elif name == "MAXITER":
            maxiter = int(val)
        elif name == "TAU":
            tau = float(val)
        elif name == "DUALVARS":
            M, N = g.shape
            val = np.asarray(val, dtype=np.float64)
            if val.shape[0] != M or val.shape[1] != 2 * N:
                raise ValueError("Wrong size of the dual variables")       # :102-104
            dual = (val[:, :M], val[:, M:])                                 # :105-107
    if maxiter is None:
        raise NameError("Undefined function or variable 'MaxIter'")        # Q4
    f, px, py, _, _ = _tv_engine(g.shape).tvprox(g, lam, maxiter, tol, tau, dual)
    return f, px, py


# ---------------------------------------------------------------------------
# closure families of the demo scripts
# ---------------------------------------------------------------------------
def _closures(model, im_size, psf_size, phi=0.0):
    eng = engine_for(im_size, psf_size, model, phi)
    A = lambda x, *psi: eng.blur(x, psi, OP_A)
    AT = lambda x, *psi: eng.blur(x, psi, OP_AT)
    d0 = lambda x, *psi: eng.blur(x, psi, OP_D0)
    d1 = lambda x, *psi: eng.blur(x, psi, OP_D1)
    H = lambda *psi: eng.psf_spectrum(psi, K_PSF)
    return dict(A=A, AT=AT, dif=(d0, d1) if model != LAPLACE else (d0,), H_FFT=H,
                HC_FFT=lambda *psi: np.conj(H(*psi)), engine=eng)


def gaussian_closures(im_size, psf_size, phi):
    """A, AT, dif_w1, dif_w2 of run_Gaussian_demo.m:126-139."""
    return _closures(GAUSSIAN, im_size, psf_size, phi)


def moffat_closures(im_size, psf_size):
    """A, AT, diff_A_alpha, diff_A_beta of run_moffat_demo.m:122-137."""
    return _closures(MOFFAT, im_size, psf_size)


def laplace_closures(im_size, psf_size):
    """A, AT, diff_A_b of run_laplace_demo.m:96-107."""
    return _closures(LAPLACE, im_size, psf_size)


# ---------------------------------------------------------------------------
# SAPG drivers
# ---------------------------------------------------------------------------
_NAMES = {GAUSSIAN: ("w1", "w2"), MOFFAT: ("alpha", "beta"), LAPLACE: ("b",)}


def make_params(model, op, c=None, n_chains=1, seed=1, chain_offset=0, total_chains=None,
                post_mean=False):
    """Flatten the MATLAB `op` (+ `c`) structs into the POD the C ABI takes."""
    p = sbd_params()
    names = _NAMES[model]
    p.samples = int(op["samples"]); p.warmup = int(op.get("warmup", 100)); p.burnIn = int(op["burnIn"])
    p.n_chains = int(n_chains)
    if model == GAUSSIAN:
        p.gam = c["gam"] * op["gamma"]; p.lamb = c["lam"] * op["lambda"]        # Guassian.m:30-31
        p.c_theta = c["theta"]; p.c_sigma2 = c["sigma"]
        cps = (c["w1"], c["w2"])
        p.sigma2_fixed = op["sigma_init"]                                       # Guassian.m:190 (Q15)
        p.err_psf_lag = 1                                                       # Guassian.m:203 (Q9)
    else:
        p.gam = op["gamma"]; p.lamb = op["lambda"]
        if model == MOFFAT:
            p.c_theta, cps, p.c_sigma2 = 0.1, (10.0, 10000.0), 10000.0          # moffat.m:135-138
        else:
            p.c_theta, cps, p.c_sigma2 = 0.01, (100.0,), 10000.0                # laplace.m:139-141
        p.sigma2_fixed = op["sigma"] ** 2                                       # moffat.m:197 (Q15)
        p.err_psf_lag = 0
    p.prox_lambda = op["lambda"]                                                # run_Gaussian_demo.m:191
    p.chambolle_maxiter = int(op.get("chambolleit", 25))
    p.chambolle_tol = 1e-3; p.chambolle_tau = 0.249
    p.th_init = op["th_init"]; p.min_th = op["min_th"]; p.max_th = op["max_th"]
    for i, n in enumerate(names):
        p.psi_init[i] = op[n + "_init"]; p.psi_min[i] = op["min_" + n]; p.psi_max[i] = op["max_" + n]
        p.c_psi[i] = cps[i]; p.psi_fixed[i] = op[n]; p.psi_true[i] = op[n]; p.fix_psi[i] = int(bool(op["fix_" + n]))
    p.sigma2_init = op["sigma_init"]; p.sigma2_min = op["sigma_min"]; p.sigma2_max = op["sigma_max"]
    p.fix_sigma = int(bool(op["fix_sigma"]))
    p.d_scale = op["d_scale"]; p.d_exp = op["d_exp"]
    p.seed = int(seed); p.chain_offset = int(chain_offset)
    p.total_chains = int(total_chains if total_chains is not None else n_chains)
    p.post_mean = int(bool(post_mean)); p.use_graph = int(op.get("use_graph", -1))       # -1: automatic
    return p


def _run(model, y, op, c, noise=None, n_chains=1, seed=1, engine=None, post_mean=False, x_true=None, post_levels=0,
         post_batch=0):
    if int(post_batch) < -1:
        raise ValueError(f"post_batch must be 0 (off), -1 (floor(sqrt(n))) or a batch length >= 1, got {post_batch}")
    y = np.asarray(y, dtype=np.float64)
    op = dict(op)
    if "warmup" not in op:
        op["warmup"] = 100                                                      # Guassian.m:19-21
    prm = make_params(model, op, c, n_chains=n_chains, seed=seed, post_mean=post_mean)
    eng = engine or engine_for(y.shape, op["psf_size"], model, op.get("phi", 0.0), max_batch=n_chains)
    X0 = op.get("X0")                                                           # Guassian.m:10-12
    out = eng.sapg(y, prm, X0=X0, x_true=x_true, noise=noise, want_X_mean=post_mean, post_levels=post_levels,
                   post_batch=post_batch)
    return op, prm, out


def _add_posterior(r, o):
    """results.posterior (one dict per block size) and, at the pixel scale, posteriorvar / posteriorstd / Rhat -
    only when the statistics were requested, so that the default results keep the reference's field set."""
    if "posterior" in o:
        p0 = o["posterior"][0]
        r.update(posterior=o["posterior"], posteriorvar=p0["var"], posteriorstd=p0["std"], Rhat=p0["Rhat"])
        if "ESS" in p0:                         # post_batch
            r.update(ESS=p0["ESS"], MCSE=p0["MCSE"], Rhat_split=p0["Rhat_split"])
    return r


def SAPG_algorithm_Guassian(y, op, c, noise=None, n_chains=1, seed=1, engine=None, post_mean=False, post_levels=0,
                            post_batch=0):
    """[theta_EB, w1_EB, w2_EB, sigma_EB, results] = SAPG_algorithm_Guassian(y, op, c)
    SAPG/SAPG_algorithm_Guassian.m:7-308.  `op` must carry the plain-data fields
    the reference already stores (psf_size, phi, lambda, gamma, ...); the function
    handles in `op` are not used - the engine implements the model they encode.  post_levels > 0 adds the posterior
    statistics (Engine.sapg) as results["posterior"], ["posteriorvar"], ["posteriorstd"], ["Rhat"]; post_batch
    (-1 or b >= 1, with post_levels) adds the pixel-scale results["ESS"], ["MCSE"], ["Rhat_split"]."""
    op, prm, o = _run(GAUSSIAN, y, op, c, noise, n_chains, seed, engine, post_mean, post_levels=post_levels,
                      post_batch=post_batch)
    r = dict(logPiTrace_WU=o["logPiTrace_WU"], execTimeFindParameters=o["seconds"], last_samp=o["last_samp"],
             logPiTraceX=o["logPiTraceX"], gXTrace=o["gXTrace"],
             theta_EB=o["EB"][0], last_theta=o["thetas"][-1], thetas=o["thetas"], mean_thetas=o["mean_theta"],
             tol_thetas=o["tol_theta"],
             w1_EB=o["EB"][1], last_w1=o["psi0"][-1], w1s=o["psi0"], mean_w1s=o["mean_psi0"], tol_w1s=o["tol_psi0"],
             w2_EB=o["EB"][2], last_w2=o["psi1"][-1], w2s=o["psi1"], mean_w2s=o["mean_psi1"], tol_w2s=o["tol_psi1"],
             sigma_EB=o["EB"][3], last_sigma=o["sigmas"][-1], sigmas=o["sigmas"], mean_sigmas=o["mean_sigma"],
             tol_sigma=o["tol_sigma"], c_theta=c["theta"], c_w1=c["w1"], c_w2=c["w2"], c_sigma=c["sigma"],
             Xlast_sample=o["X_last"][0] if n_chains == 1 else o["X_last"], err_psf=o["err_psf"],
             grad_theta=o["grad_theta"], grad_w1=o["grad_psi0"], grad_w2=o["grad_psi1"],
             grad_sigma=o["grad_sigma"], options=op,
             chambolle_iters=o["chambolle_iters"], X_warm=o.get("X_warm"), posteriormean=o.get("X_mean"))
    _add_posterior(r, o)
    return r["theta_EB"], r["w1_EB"], r["w2_EB"], r["sigma_EB"], r


def SAPG_algorithm_moffat(y, op, noise=None, n_chains=1, seed=1, engine=None, post_mean=False, post_levels=0,
                          post_batch=0):
    """[theta_EB, alpha_EB, beta_EB, sigma2_EB, results] = SAPG_algorithm_moffat(y, op)
    SAPG/SAPG_algorithm_moffat.m:7-297."""
    op, prm, o = _run(MOFFAT, y, op, None, noise, n_chains, seed, engine, post_mean, post_levels=post_levels,
                      post_batch=post_batch)
    err_psf = o["err_psf"].copy(); err_psf[0] = 0.0          # err_psf(1) is never assigned (moffat.m:205)
    r = {"lambda": op["lambda"], "gamma": op["gamma"]}
    r.update(logPiTrace_WU=o["logPiTrace_WU"], execTimeFindTheta=o["seconds"], last_samp=o["last_samp"],
             logPiTraceX=o["logPiTraceX"], gXTrace=o["gXTrace"],
             mean_theta=o["EB"][0], last_theta=o["thetas"][-1], thetas=o["thetas"], mean_thetas=o["mean_theta"],
             tol_thetas=o["tol_theta"], c_theta=0.1,
             alpha_EB=o["EB"][1], last_alpha=o["psi0"][-1], alphas=o["psi0"], mean_alphas=o["mean_psi0"],
             tol_alphas=o["tol_psi0"], c_alpha=10.0,
             beta_EB=o["EB"][2], last_beta=o["psi1"][-1], betas=o["psi1"], mean_betas=o["mean_psi1"],
             tol_betas=o["tol_psi1"], c_beta=10000.0,
             sigma_EB=o["EB"][3], last_sigma=o["sigmas"][-1], sigmas=o["sigmas"], mean_sigmas=o["mean_sigma"],
             tol_sigma=o["tol_sigma"], c_sigma2=10000.0,
             Xlast_sample=o["X_last"][0] if n_chains == 1 else o["X_last"],
             X_warm=o["X_warm"][0] if n_chains == 1 else o["X_warm"], options=op, err_psf=err_psf,
             chambolle_iters=o["chambolle_iters"], posteriormean=o.get("X_mean"))
    _add_posterior(r, o)
    return r["mean_theta"], r["alpha_EB"], r["beta_EB"], r["sigma_EB"], r


def SAPG_algorithm_laplace(y, op, noise=None, n_chains=1, seed=1, engine=None, post_mean=False, post_levels=0,
                           post_batch=0):
    """[theta_EB, b_EB, sigma_EB, results] = SAPG_algorithm_laplace(y, op)
    SAPG/SAPG_algorithm_laplace.m:7-268 (needs op.x, the ground truth, :28)."""
    if "x" not in op:
        raise KeyError("Reference to non-existent field 'x'.")                 # laplace.m:28
    op, prm, o = _run(LAPLACE, y, op, None, noise, n_chains, seed, engine, post_mean, x_true=op["x"],
                      post_levels=post_levels, post_batch=post_batch)
    err_warm = np.zeros(max(int(op["warmup"]), 1)); err_warm[0] = o["err_warm0"]    # laplace.m:28-29
    r = {"lambda": op["lambda"], "gamma": op["gamma"]}
    r.update(logPiTrace_WU=o["logPiTrace_WU"], execTimeFindTheta=o["seconds"], last_samp=o["last_samp"],
             logPiTraceX=o["logPiTraceX"], gXTrace=o["gXTrace"],
             mean_theta=o["EB"][0], last_theta=o["thetas"][-1], thetas=o["thetas"], mean_thetas=o["mean_theta"],
             tol_thetas=o["tol_theta"], c_theta=0.01,
             mean_b=o["EB"][1], last_b=o["psi0"][-1], bs=o["psi0"], mean_bs=o["mean_psi0"], tol_bs=o["tol_psi0"],
             c_b=100.0,
             sigma_EB=o["EB"][3], last_sigma=o["sigmas"][-1], sigmas=o["sigmas"], mean_sigmas=o["mean_sigma"],
             tol_sigma=o["tol_sigma"], c_sigma2=10000.0,
             X_sample=o["X_last"][0] if n_chains == 1 else o["X_last"],
             X_warm=o["X_warm"][0] if n_chains == 1 else o["X_warm"],
             err_warm=err_warm, err_sample=o["err_sample"], err_psf=o["err_psf"], options=op,
             chambolle_iters=o["chambolle_iters"], posteriormean=o.get("X_mean"))
    _add_posterior(r, o)
    return r["mean_theta"], r["mean_b"], r["sigma_EB"], r
