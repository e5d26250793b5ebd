/*
 * sbd_mex.c - thin MEX gateway between MATLAB / Octave and libsbd.so.
 *
 *   out = sbd_mex(command, args...)
 *
 * It only validates and forwards: every numerical result comes from the CUDA
 * kernels behind the C ABI in include/sbd.h.  MATLAB arrays are column-major
 * doubles, which is exactly the layout the ABI takes, so no data is rearranged.
 * Contexts (one per image size / PSF family) persist behind mexLock and are
 * destroyed by the mexAtExit hook.
 *
 * Commands (the .m wrappers in ../matlab call these):
 *   tv      = sbd_mex('tvnorm', x)                                        utils/TVnorm.m
 *   d       = sbd_mex('diff', x, axis)                                    SALSA/diffh.m, diffv.m
 *   [f,px,py,k,err] = sbd_mex('tvprox', g, lambda, maxiter, tol, tau, px0, py0)
 *                                                                         utils/chambolle_prox_TV_stop.m
 *   k       = sbd_mex('psf', model, t, phi, psi, which)                   utils/psf_gaussian.m ...
 *   H       = sbd_mex('spectrum', [M N], model, t, phi, psi, which)       utils/resize.m + diff_*.m
 *   out     = sbd_mex('blur', x, model, t, phi, psi, op)                  A / AT / dif_* closures
 *   s       = sbd_mex('likelihood', x, y, model, t, phi, psi, sigma2, theta)   op.f, op.gradF, op.grad_psi, ...
 *   r       = sbd_mex('sapg', y, X0, xtrue, model, t, phi, P, noise)      SAPG/SAPG_algorithm_*.m
 *             P.post_levels = L (optional, 0 = off) adds r.posterior: a 1x1 struct with one field per block size,
 *             s1, s2, s4, ..., each a struct with scale, n, chains, mean, within, between, var, std, Rhat
 *             (include/sbd.h sbd_posterior_stats; the .m wrappers turn it into a struct array).
 *             P.post_batch = b (optional, 0 = off; -1: floor(sqrt(n)), b >= 1: batch length b; needs post_levels)
 *             adds batch_mean, batch_within, batch_between, half_mean, half_within, half_between, batch_len,
 *             n_batches, half_n, ESS, MCSE, Rhat_split to each (sbd_posterior_diagnostics)
 *             P.post_ci = alpha (optional, 0 = off; 0 < alpha < 1; needs post_levels) adds ci_alpha, ci_count, lower,
 *             median, upper, ci_width (the 1 - alpha credible interval and the median, sbd_posterior_quantiles)
 *   [v,k]   = sbd_mex('max_eigenval', [M N], model, t, phi, psi, tol, maxit, x0)   utils/max_eigenval_*.m
 *   [y,s,n] = sbd_mex('observe', x, model, t, phi, psi, bsnr, noise)      run_Gaussian_demo.m:145-168
 *   [x,obj,dist,mses] = sbd_mex('salsa', y, model, t, phi, psi, tau, mu, maxiter, tolA, tviters, xtrue)
 *                                                                         SALSA/SALSA_v2.m as the demos call it
 *
 * Build:  mex -I../../include sbd_mex.c -L../lib -lsbd          (MATLAB)
 *         mkoctfile --mex -I../../include sbd_mex.c -L../lib -lsbd   (Octave)
 */
#include <math.h>
#include <string.h>
#include <stdio.h>
#include "mex.h"
#include "sbd.h"

#define MAX_CTX 16
typedef struct { sbd_ctx* h; int rows, cols, t, model, batch; double phi; } ctx_slot;
static ctx_slot g_ctx[MAX_CTX];
static int g_nctx = 0, g_locked = 0;

static void cleanup(void) {
    int i;
    for (i = 0; i < g_nctx; ++i) sbd_destroy(g_ctx[i].h);
    g_nctx = 0;
}

static void fail(sbd_ctx* c, const char* where, int rc) {
    mexErrMsgIdAndTxt("sbd:error", "%s failed (%d): %s", where, rc, sbd_last_error(c));
}

static sbd_ctx* get_ctx(int rows, int cols, int t, int model, double phi, int batch) {
    int i, rc;
    sbd_ctx* h = NULL;
    for (i = 0; i < g_nctx; ++i) {
        ctx_slot* s = &g_ctx[i];
        if (s->rows == rows && s->cols == cols && s->t == t && s->model == model && s->phi == phi &&
            s->batch >= batch)
            return s->h;
    }
    if (g_nctx == MAX_CTX) { cleanup(); }
    rc = sbd_create(&h, rows, cols, t, model, phi, batch, 0);
    if (rc != SBD_OK) fail(NULL, "sbd_create", rc);
    if (!g_locked) { mexLock(); mexAtExit(cleanup); g_locked = 1; }
    g_ctx[g_nctx].h = h; g_ctx[g_nctx].rows = rows; g_ctx[g_nctx].cols = cols; g_ctx[g_nctx].t = t;
    g_ctx[g_nctx].model = model; g_ctx[g_nctx].phi = phi; g_ctx[g_nctx].batch = batch;
    ++g_nctx;
    return h;
}

static const double* image(const mxArray* a, const char* name, int* rows, int* cols) {
    if (!mxIsDouble(a) || mxIsComplex(a) || mxGetNumberOfDimensions(a) != 2)
        mexErrMsgIdAndTxt("sbd:type", "%s must be a real double matrix", name);
    *rows = (int)mxGetM(a); *cols = (int)mxGetN(a);
    return mxGetPr(a);
}

static void psi_of(const mxArray* a, double psi[2]) {
    size_t n = mxGetNumberOfElements(a);
    psi[0] = n > 0 ? mxGetPr(a)[0] : 0.0;
    psi[1] = n > 1 ? mxGetPr(a)[1] : 0.0;
}

static double field(const mxArray* s, const char* name, int required, double dflt) {
    const mxArray* f = mxGetField(s, 0, name);
    if (!f || mxIsEmpty(f)) {
        if (required) mexErrMsgIdAndTxt("sbd:field", "Reference to non-existent field '%s'.", name);
        return dflt;
    }
    return mxGetScalar(f);
}

static void field2(const mxArray* s, const char* name, double out[2]) {
    const mxArray* f = mxGetField(s, 0, name);
    out[0] = out[1] = 0.0;
    if (f) psi_of(f, out);
}

static mxArray* vec(int n, double** p) {
    mxArray* a = mxCreateDoubleMatrix(1, n > 0 ? n : 0, mxREAL);
    *p = mxGetPr(a);
    return a;
}

/* posterior statistics of the last run at block sizes 1 .. 2^(levels-1), with var, std and Rhat formed as DESIGN.md
   states them ("Posterior statistics"); diag: also the diagnostics with ESS, MCSE and Rhat_split; ci: also the
   credible interval and the median */
static mxArray* posterior_struct(sbd_ctx* c, int rows, int cols, int levels, int diag, int ci) {
    static const char* fields[] = {"scale", "n", "chains", "mean", "within", "between", "var", "std", "Rhat",
                                   "batch_mean", "batch_within", "batch_between", "half_mean", "half_within",
                                   "half_between", "batch_len", "n_batches", "half_n", "ESS", "MCSE", "Rhat_split"};
    static const char* qfields[] = {"ci_alpha", "ci_count", "lower", "median", "upper", "ci_width"};
    const char* names[27];
    char lnames[8][8];
    const char* lp[8];
    mxArray* out;
    int j, rc, nf = 0;
    for (j = 0; j < (diag ? 21 : 9); ++j) names[nf++] = fields[j];
    for (j = 0; ci && j < 6; ++j) names[nf++] = qfields[j];
    for (j = 0; j < levels; ++j) { snprintf(lnames[j], sizeof lnames[j], "s%d", 1 << j); lp[j] = lnames[j]; }
    out = mxCreateStructMatrix(1, 1, levels, lp);
    for (j = 0; j < levels; ++j) {
        const int s = 1 << j, bx = (rows + s - 1) / s, by = (cols + s - 1) / s;
        mxArray* e = mxCreateStructMatrix(1, 1, nf, names);
        mxArray *a[6];
        double* p[6];
        int q, n = 0, C = 0;
        size_t i;
        for (q = 0; q < 6; ++q) { a[q] = mxCreateDoubleMatrix(bx, by, mxREAL); p[q] = mxGetPr(a[q]); }
        rc = sbd_posterior_stats(c, j, p[0], p[1], p[2], &n, &C);
        if (rc) { sbd_set_posterior(c, 0); fail(c, "sbd_posterior_stats", rc); }
        for (i = 0; i < (size_t)bx * by; ++i) {
            const double W = p[1][i], B = p[2][i];
            p[3][i] = C * n >= 2 ? (W + n * B) / (double)(C * n - 1) : NAN;            /* var */
            p[4][i] = sqrt(p[3][i]);                                                 /* std */
            p[5][i] = (C >= 2 && n >= 2)                                             /* Gelman-Rubin Rhat */
                ? sqrt(((n - 1.0) / n * (W / (C * (n - 1.0))) + B / (C - 1.0)) / (W / (C * (n - 1.0)))) : NAN;
        }
        mxSetField(e, 0, "scale", mxCreateDoubleScalar((double)s));
        mxSetField(e, 0, "n", mxCreateDoubleScalar((double)n));
        mxSetField(e, 0, "chains", mxCreateDoubleScalar((double)C));
        mxSetField(e, 0, "mean", a[0]); mxSetField(e, 0, "within", a[1]); mxSetField(e, 0, "between", a[2]);
        mxSetField(e, 0, "var", a[3]); mxSetField(e, 0, "std", a[4]); mxSetField(e, 0, "Rhat", a[5]);
        if (diag) {
            mxArray* d[9];
            double* g[9];
            int b = 0, B = 0, h = 0;
            for (q = 0; q < 9; ++q) { d[q] = mxCreateDoubleMatrix(bx, by, mxREAL); g[q] = mxGetPr(d[q]); }
            rc = sbd_posterior_diagnostics(c, j, g[0], g[1], g[2], g[3], g[4], g[5], &b, &B, &h);
            if (rc) { sbd_set_posterior(c, 0); sbd_set_posterior_diagnostics(c, 0); fail(c, "sbd_posterior_diagnostics", rc); }
            for (i = 0; i < (size_t)bx * by; ++i) {
                const double tau2 = C * B >= 2 ? b * (g[1][i] + B * g[2][i]) / (C * (double)B - 1.0) : NAN;
                const double Wh = g[4][i] / (2.0 * C * (h - 1.0)), Bh = g[5][i] / (2.0 * C - 1.0);
                g[6][i] = C * (double)n * p[3][i] / tau2;                                /* ESS */
                g[7][i] = sqrt(tau2 / (C * (double)n));                                  /* MCSE */
                g[8][i] = h >= 2 ? sqrt(((h - 1.0) / h * Wh + Bh) / Wh) : NAN;           /* split Rhat */
            }
            for (q = 0; q < 6; ++q) mxSetField(e, 0, fields[9 + q], d[q]);
            mxSetField(e, 0, "batch_len", mxCreateDoubleScalar((double)b));
            mxSetField(e, 0, "n_batches", mxCreateDoubleScalar((double)B));
            mxSetField(e, 0, "half_n", mxCreateDoubleScalar((double)h));
            mxSetField(e, 0, "ESS", d[6]); mxSetField(e, 0, "MCSE", d[7]); mxSetField(e, 0, "Rhat_split", d[8]);
        }
        if (ci) {
            mxArray* u[4];
            double* g[4];
            double alpha = 0.0;
            long long count = 0;
            for (q = 0; q < 4; ++q) { u[q] = mxCreateDoubleMatrix(bx, by, mxREAL); g[q] = mxGetPr(u[q]); }
            rc = sbd_posterior_quantiles(c, j, g[0], g[1], g[2], &alpha, &count);
            if (rc) {
                sbd_set_posterior(c, 0); sbd_set_posterior_diagnostics(c, 0); sbd_set_posterior_quantiles(c, 0.0);
                fail(c, "sbd_posterior_quantiles", rc);
            }
            for (i = 0; i < (size_t)bx * by; ++i) g[3][i] = g[2][i] - g[0][i];         /* ci_width */
            mxSetField(e, 0, "ci_alpha", mxCreateDoubleScalar(alpha));
            mxSetField(e, 0, "ci_count", mxCreateDoubleScalar((double)count));
            mxSetField(e, 0, "lower", u[0]); mxSetField(e, 0, "median", u[1]); mxSetField(e, 0, "upper", u[2]);
            mxSetField(e, 0, "ci_width", u[3]);
        }
        mxSetField(out, 0, lp[j], e);
    }
    return out;
}

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    char cmd[32];
    int rows, cols, rc;
    if (nrhs < 1 || !mxIsChar(prhs[0]) || mxGetString(prhs[0], cmd, sizeof cmd))
        mexErrMsgIdAndTxt("sbd:usage", "sbd_mex(command, ...)");

    if (!strcmp(cmd, "tvnorm")) {
        const double* x = image(prhs[1], "x", &rows, &cols);
        sbd_ctx* c = get_ctx(rows, cols, 1, SBD_GAUSSIAN, 0.0, 1);
        double v = 0.0;
        if ((rc = sbd_tvnorm(c, x, &v, 1))) fail(c, "sbd_tvnorm", rc);
        plhs[0] = mxCreateDoubleScalar(v);
    } else if (!strcmp(cmd, "diff")) {
        const double* x = image(prhs[1], "x", &rows, &cols);
        sbd_ctx* c = get_ctx(rows, cols, 1, SBD_GAUSSIAN, 0.0, 1);
        plhs[0] = mxCreateDoubleMatrix(rows, cols, mxREAL);
        if ((rc = sbd_diff(c, x, (int)mxGetScalar(prhs[2]), mxGetPr(plhs[0]), 1))) fail(c, "sbd_diff", rc);
    } else if (!strcmp(cmd, "tvprox")) {
        const double* g = image(prhs[1], "g", &rows, &cols);
        sbd_ctx* c = get_ctx(rows, cols, 1, SBD_GAUSSIAN, 0.0, 1);
        const double *px0 = NULL, *py0 = NULL;
        int r2, c2, iters = 0;
        double err = 0.0;
        mxArray *f = mxCreateDoubleMatrix(rows, cols, mxREAL), *px = mxCreateDoubleMatrix(rows, cols, mxREAL),
                *py = mxCreateDoubleMatrix(rows, cols, mxREAL);
        if (nrhs > 7 && !mxIsEmpty(prhs[6])) {
            px0 = image(prhs[6], "px", &r2, &c2);
            if (r2 != rows || c2 != cols) mexErrMsgIdAndTxt("sbd:size", "Wrong size of the dual variables");
            py0 = image(prhs[7], "py", &r2, &c2);
            if (r2 != rows || c2 != cols) mexErrMsgIdAndTxt("sbd:size", "Wrong size of the dual variables");
        }
        rc = sbd_tvprox(c, g, mxGetScalar(prhs[2]), (int)mxGetScalar(prhs[3]), mxGetScalar(prhs[4]),
                        mxGetScalar(prhs[5]), px0, py0, mxGetPr(f), mxGetPr(px), mxGetPr(py), &iters, &err, 1);
        if (rc) fail(c, "sbd_tvprox", rc);
        plhs[0] = f;
        if (nlhs > 1) plhs[1] = px;
        if (nlhs > 2) plhs[2] = py;
        if (nlhs > 3) plhs[3] = mxCreateDoubleScalar((double)iters);
        if (nlhs > 4) plhs[4] = mxCreateDoubleScalar(err);
    } else if (!strcmp(cmd, "psf")) {
        const int model = (int)mxGetScalar(prhs[1]), t = (int)mxGetScalar(prhs[2]);
        double psi[2];
        sbd_ctx* c = get_ctx(t > 16 ? t : 16, t > 16 ? t : 16, t, model, mxGetScalar(prhs[3]), 1);
        psi_of(prhs[4], psi);
        plhs[0] = mxCreateDoubleMatrix(t, t, mxREAL);
        if ((rc = sbd_psf_taps(c, psi, (int)mxGetScalar(prhs[5]), mxGetPr(plhs[0])))) fail(c, "sbd_psf_taps", rc);
    } else if (!strcmp(cmd, "spectrum")) {
        const double* sz = mxGetPr(prhs[1]);
        double psi[2];
        sbd_ctx* c;
        rows = (int)sz[0]; cols = (int)sz[1];
        c = get_ctx(rows, cols, (int)mxGetScalar(prhs[3]), (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[4]), 1);
        psi_of(prhs[5], psi);
        plhs[0] = mxCreateDoubleMatrix(rows, cols, mxCOMPLEX);
        rc = sbd_psf_spectrum(c, psi, (int)mxGetScalar(prhs[6]), mxGetPr(plhs[0]), mxGetPi(plhs[0]));
        if (rc) fail(c, "sbd_psf_spectrum", rc);
    } else if (!strcmp(cmd, "blur")) {
        const double* x = image(prhs[1], "x", &rows, &cols);
        double psi[2];
        sbd_ctx* c = get_ctx(rows, cols, (int)mxGetScalar(prhs[3]), (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[4]), 1);
        psi_of(prhs[5], psi);
        plhs[0] = mxCreateDoubleMatrix(rows, cols, mxREAL);
        if ((rc = sbd_blur(c, x, psi, (int)mxGetScalar(prhs[6]), mxGetPr(plhs[0]), 1))) fail(c, "sbd_blur", rc);
    } else if (!strcmp(cmd, "likelihood")) {
        const double* x = image(prhs[1], "x", &rows, &cols);
        int r2, c2;
        const double* y = image(prhs[2], "y", &r2, &c2);
        double psi[2], *s;
        mxArray* gf = mxCreateDoubleMatrix(rows, cols, mxREAL);
        sbd_ctx* c = get_ctx(rows, cols, (int)mxGetScalar(prhs[4]), (int)mxGetScalar(prhs[3]), mxGetScalar(prhs[5]), 1);
        if (r2 != rows || c2 != cols) mexErrMsgIdAndTxt("sbd:size", "x and y differ in size");
        psi_of(prhs[6], psi);
        plhs[0] = vec(6, &s);
        rc = sbd_likelihood(c, x, y, psi, mxGetScalar(prhs[7]), mxGetScalar(prhs[8]), s, mxGetPr(gf));
        if (rc) fail(c, "sbd_likelihood", rc);
        if (nlhs > 1) plhs[1] = gf;
    } else if (!strcmp(cmd, "sapg")) {
        /* r = sbd_mex('sapg', y, X0, xtrue, model, t, phi, P, noise) ; P = struct of sbd_params fields */
        static const char* names[] = {"logPiTrace_WU", "thetas", "sigmas", "psi0", "psi1", "grad_theta", "grad_psi0",
                                      "grad_psi1", "grad_sigma", "logPiTraceX", "gXTrace", "err_psf", "err_sample",
                                      "tol_theta", "tol_psi0", "tol_psi1", "tol_sigma", "mean_theta", "mean_psi0",
                                      "mean_psi1", "mean_sigma", "X_warm", "X_last", "EB", "err_warm0", "seconds",
                                      "last_samp", "posterior"};
        const double* y = image(prhs[1], "y", &rows, &cols);
        const double* X0 = mxIsEmpty(prhs[2]) ? NULL : mxGetPr(prhs[2]);
        const double* xt = mxIsEmpty(prhs[3]) ? NULL : mxGetPr(prhs[3]);
        const mxArray* P = prhs[7];
        const double* noise = (nrhs > 8 && !mxIsEmpty(prhs[8])) ? mxGetPr(prhs[8]) : NULL;
        sbd_params p;
        sbd_traces t;
        sbd_ctx* c;
        double* q[21];
        int i, nm, levels, batch;
        double ci;
        mxArray* r;
        if (!mxIsStruct(P)) mexErrMsgIdAndTxt("sbd:type", "P must be a struct");
        memset(&p, 0, sizeof p); memset(&t, 0, sizeof t);
        p.samples = (int)field(P, "samples", 1, 0); p.warmup = (int)field(P, "warmup", 0, 100);
        p.burnIn = (int)field(P, "burnIn", 1, 0); p.n_chains = (int)field(P, "n_chains", 0, 1);
        p.gam = field(P, "gam", 1, 0); p.lamb = field(P, "lamb", 1, 0); p.prox_lambda = field(P, "prox_lambda", 1, 0);
        p.chambolle_maxiter = (int)field(P, "chambolle_maxiter", 0, 25);
        p.chambolle_tol = field(P, "chambolle_tol", 0, 1e-3); p.chambolle_tau = field(P, "chambolle_tau", 0, 0.249);
        p.th_init = field(P, "th_init", 1, 0); p.min_th = field(P, "min_th", 1, 0); p.max_th = field(P, "max_th", 1, 0);
        p.c_theta = field(P, "c_theta", 1, 0);
        field2(P, "psi_init", p.psi_init); field2(P, "psi_min", p.psi_min); field2(P, "psi_max", p.psi_max);
        field2(P, "c_psi", p.c_psi); field2(P, "psi_fixed", p.psi_fixed); field2(P, "psi_true", p.psi_true);
        { double fx[2]; field2(P, "fix_psi", fx); p.fix_psi[0] = fx[0] != 0; p.fix_psi[1] = fx[1] != 0; }
        p.sigma2_init = field(P, "sigma2_init", 1, 0); p.sigma2_min = field(P, "sigma2_min", 1, 0);
        p.sigma2_max = field(P, "sigma2_max", 1, 0); p.c_sigma2 = field(P, "c_sigma2", 1, 0);
        p.sigma2_fixed = field(P, "sigma2_fixed", 0, 0); p.fix_sigma = (int)field(P, "fix_sigma", 0, 0);
        p.err_psf_lag = (int)field(P, "err_psf_lag", 0, 0);
        p.d_scale = field(P, "d_scale", 1, 0); p.d_exp = field(P, "d_exp", 1, 0);
        p.seed = (uint64_t)field(P, "seed", 0, 1); p.chain_offset = 0; p.total_chains = p.n_chains;
        p.use_graph = (int)field(P, "use_graph", 0, -1);            /* -1: automatic (CUDA graph for small problems) */
        levels = (int)field(P, "post_levels", 0, 0);                 /* posterior statistics, 0 = off */
        batch = (int)field(P, "post_batch", 0, 0);                   /* their diagnostics, 0 = off */
        ci = field(P, "post_ci", 0, 0);                              /* credible level alpha, 0 = off */
        c = get_ctx(rows, cols, (int)mxGetScalar(prhs[5]), (int)mxGetScalar(prhs[4]), mxGetScalar(prhs[6]), p.n_chains);
        nm = p.samples - p.burnIn; if (nm < 0) nm = 0;
        /* the `posterior` field exists only when it was asked for: otherwise the old field set */
        r = mxCreateStructMatrix(1, 1, (int)(sizeof names / sizeof names[0]) - (levels > 0 ? 0 : 1), names);
        for (i = 0; i < 21; ++i) {
            const int len = (i == 0) ? p.warmup : (i >= 17 ? nm : p.samples);
            mxSetField(r, 0, names[i], vec(len, &q[i]));
        }
        t.logPiTrace_WU = q[0]; t.thetas = q[1]; t.sigmas = q[2]; t.psi0 = q[3]; t.psi1 = q[4];
        t.grad_theta = q[5]; t.grad_psi0 = q[6]; t.grad_psi1 = q[7]; t.grad_sigma = q[8];
        t.logPiTraceX = q[9]; t.gXTrace = q[10]; t.err_psf = q[11]; t.err_sample = q[12];
        t.tol_theta = q[13]; t.tol_psi0 = q[14]; t.tol_psi1 = q[15]; t.tol_sigma = q[16];
        t.mean_theta = q[17]; t.mean_psi0 = q[18]; t.mean_psi1 = q[19]; t.mean_sigma = q[20];
        { mxArray* a = mxCreateDoubleMatrix(rows, cols * p.n_chains, mxREAL); t.X_warm = mxGetPr(a); mxSetField(r, 0, "X_warm", a); }
        { mxArray* a = mxCreateDoubleMatrix(rows, cols * p.n_chains, mxREAL); t.X_last = mxGetPr(a); mxSetField(r, 0, "X_last", a); }
        if ((rc = sbd_set_posterior(c, levels))) fail(c, "sbd_set_posterior", rc);
        if ((rc = sbd_set_posterior_diagnostics(c, batch))) { sbd_set_posterior(c, 0); fail(c, "sbd_set_posterior_diagnostics", rc); }
        if ((rc = sbd_set_posterior_quantiles(c, ci))) {
            sbd_set_posterior(c, 0); sbd_set_posterior_diagnostics(c, 0); fail(c, "sbd_set_posterior_quantiles", rc);
        }
        rc = sbd_sapg_run(c, y, X0, xt, &p, noise, &t);
        if (rc) {
            sbd_set_posterior(c, 0); sbd_set_posterior_diagnostics(c, 0); sbd_set_posterior_quantiles(c, 0.0);
            fail(c, "sbd_sapg_run", rc);
        }
        if (levels > 0) {
            mxArray* post;
            post = posterior_struct(c, rows, cols, levels, batch != 0, ci != 0.0);
            sbd_set_posterior(c, 0);                             /* cached context: the requests are sticky */
            sbd_set_posterior_diagnostics(c, 0);
            sbd_set_posterior_quantiles(c, 0.0);
            mxSetField(r, 0, "posterior", post);
        }
        { double* e; mxSetField(r, 0, "EB", vec(4, &e)); for (i = 0; i < 4; ++i) e[i] = t.EB[i]; }
        mxSetField(r, 0, "err_warm0", mxCreateDoubleScalar(t.err_warm0));
        mxSetField(r, 0, "seconds", mxCreateDoubleScalar(t.seconds));
        mxSetField(r, 0, "last_samp", mxCreateDoubleScalar((double)t.last_samp));
        plhs[0] = r;
    } else if (!strcmp(cmd, "max_eigenval")) {
        const double* sz = mxGetPr(prhs[1]);
        double psi[2], val = 0.0;
        int it = 0;
        sbd_ctx* c;
        const double* x0 = (nrhs > 8 && !mxIsEmpty(prhs[8])) ? mxGetPr(prhs[8]) : NULL;
        rows = (int)sz[0]; cols = (int)sz[1];
        c = get_ctx(rows, cols, (int)mxGetScalar(prhs[3]), (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[4]), 1);
        psi_of(prhs[5], psi);
        rc = sbd_max_eigenval(c, psi, x0, mxGetScalar(prhs[6]), (int)mxGetScalar(prhs[7]), 1, &val, &it);
        if (rc) fail(c, "sbd_max_eigenval", rc);
        plhs[0] = mxCreateDoubleScalar(val);
        if (nlhs > 1) plhs[1] = mxCreateDoubleScalar((double)it);
    } else if (!strcmp(cmd, "observe")) {
        const double* x = image(prhs[1], "x", &rows, &cols);
        double psi[2], sg = 0.0, nr = 0.0;
        const double* noise = (nrhs > 7 && !mxIsEmpty(prhs[7])) ? mxGetPr(prhs[7]) : NULL;
        sbd_ctx* c = get_ctx(rows, cols, (int)mxGetScalar(prhs[3]), (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[4]), 1);
        psi_of(prhs[5], psi);
        plhs[0] = mxCreateDoubleMatrix(rows, cols, mxREAL);
        rc = sbd_observe(c, x, psi, mxGetScalar(prhs[6]), noise, 1, mxGetPr(plhs[0]), &sg, &nr);
        if (rc) fail(c, "sbd_observe", rc);
        if (nlhs > 1) plhs[1] = mxCreateDoubleScalar(sg);
        if (nlhs > 2) plhs[2] = mxCreateDoubleScalar(nr);
    } else if (!strcmp(cmd, "salsa")) {
        const double* y = image(prhs[1], "y", &rows, &cols);
        double psi[2], *obj, *dist, *ms;
        const int maxiter = (int)mxGetScalar(prhs[8]);
        const double* xt = (nrhs > 11 && !mxIsEmpty(prhs[11])) ? mxGetPr(prhs[11]) : NULL;
        int n = 0;
        mxArray *o, *d, *m;
        sbd_ctx* c = get_ctx(rows, cols, (int)mxGetScalar(prhs[3]), (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[4]), 1);
        psi_of(prhs[5], psi);
        plhs[0] = mxCreateDoubleMatrix(rows, cols, mxREAL);
        o = vec(maxiter + 1, &obj); d = vec(maxiter, &dist); m = vec(maxiter + 1, &ms);
        rc = sbd_salsa_tv(c, y, psi, mxGetScalar(prhs[6]), mxGetScalar(prhs[7]), maxiter, mxGetScalar(prhs[9]),
                          (int)mxGetScalar(prhs[10]), xt, mxGetPr(plhs[0]), obj, dist, ms, &n);
        if (rc) fail(c, "sbd_salsa_tv", rc);
        if (nlhs > 1) plhs[1] = o;
        if (nlhs > 2) plhs[2] = d;
        if (nlhs > 3) plhs[3] = m;
        if (nlhs > 4) plhs[4] = mxCreateDoubleScalar((double)n);
    } else {
        mexErrMsgIdAndTxt("sbd:usage", "unknown command '%s'", cmd);
    }
}
