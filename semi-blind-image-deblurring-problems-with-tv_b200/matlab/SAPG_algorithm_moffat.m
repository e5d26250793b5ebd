function [theta_EB, alpha_EB, beta_EB, sigma2_EB, results] = SAPG_algorithm_moffat(y, op)
% Drop-in for SAPG/SAPG_algorithm_moffat.m:7-297 - same signature, same `results` fields.
P = sbd_pack(1, op, []);
X0 = []; if isfield(op, 'X0'), X0 = op.X0; end
noise = []; if isfield(op, 'noise'), noise = op.noise; end
r = sbd_mex('sapg', double(y), X0, [], 1, op.psf_size, 0, P, noise);
theta_EB = r.EB(1); alpha_EB = r.EB(2); beta_EB = r.EB(3); sigma2_EB = r.EB(4);
results.lambda = op.lambda; results.gamma = op.gamma;
results.logPiTrace_WU = r.logPiTrace_WU; results.execTimeFindTheta = r.seconds;
results.last_samp = r.last_samp; results.logPiTraceX = r.logPiTraceX; results.gXTrace = r.gXTrace;
results.mean_theta = theta_EB; results.last_theta = r.thetas(end); results.thetas = r.thetas;
results.mean_thetas = r.mean_theta; results.tol_thetas = r.tol_theta; results.c_theta = 0.1;
results.alpha_EB = alpha_EB; results.last_alpha = r.psi0(end); results.alphas = r.psi0;
results.mean_alphas = r.mean_psi0; results.tol_alphas = r.tol_psi0; results.c_alpha = 10;
results.beta_EB = beta_EB; results.last_beta = r.psi1(end); results.betas = r.psi1;
results.mean_betas = r.mean_psi1; results.tol_betas = r.tol_psi1; results.c_beta = 10000;
results.sigma_EB = sigma2_EB; results.last_sigma = r.sigmas(end); results.sigmas = r.sigmas;
results.mean_sigmas = r.mean_sigma; results.tol_sigma = r.tol_sigma; results.c_sigma2 = 10000;
results.Xlast_sample = r.X_last; results.X_warm = r.X_warm; results.options = op;
results.err_psf = r.err_psf; results.err_psf(1) = 0;          % err_psf(1) is never assigned (moffat.m:205)
if isfield(r, 'posterior'), results = sbd_posterior(results, r); end   % only with op.post_levels > 0
end
