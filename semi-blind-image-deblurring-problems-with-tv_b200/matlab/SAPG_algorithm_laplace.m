function [theta_EB, b_EB, sigma_EB, results] = SAPG_algorithm_laplace(y, op)
% Drop-in for SAPG/SAPG_algorithm_laplace.m:7-268 - same signature, same `results` fields
% (needs op.x, the ground truth, exactly like the reference: laplace.m:28).
P = sbd_pack(2, op, []);
X0 = []; if isfield(op, 'X0'), X0 = op.X0; end
noise = []; if isfield(op, 'noise'), noise = op.noise; end
r = sbd_mex('sapg', double(y), X0, double(op.x), 2, op.psf_size, 0, P, noise);
theta_EB = r.EB(1); b_EB = r.EB(2); sigma_EB = r.EB(4);
results.lambda = op.lambda; results.gamma = op.gamma;
results.logPiTrace_WU = r.logPiTrace_WU; results.execTimeFindTheta = r.seconds;
results.last_samp = r.last_samp; results.logPiTraceX = r.logPiTraceX; results.gXTrace = r.gXTrace;
results.mean_theta = theta_EB; results.last_theta = r.thetas(end); results.thetas = r.thetas;
results.mean_thetas = r.mean_theta; results.tol_thetas = r.tol_theta; results.c_theta = 0.01;
results.mean_b = b_EB; results.last_b = r.psi0(end); results.bs = r.psi0;
results.mean_bs = r.mean_psi0; results.tol_bs = r.tol_psi0; results.c_b = 100;
results.sigma_EB = sigma_EB; results.last_sigma = r.sigmas(end); results.sigmas = r.sigmas;
results.mean_sigmas = r.mean_sigma; results.tol_sigma = r.tol_sigma; results.c_sigma2 = 10000;
results.X_sample = r.X_last; results.X_warm = r.X_warm;
results.err_warm = zeros(1, max(op.warmup, 1)); results.err_warm(1) = r.err_warm0;   % laplace.m:28-29
results.err_sample = r.err_sample; results.err_psf = r.err_psf; results.options = op;
if isfield(r, 'posterior'), results = sbd_posterior(results, r); end   % only with op.post_levels > 0
end
