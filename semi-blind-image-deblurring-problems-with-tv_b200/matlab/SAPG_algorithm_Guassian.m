function [theta_EB, w1_EB, w2_EB, sigma_EB, results] = SAPG_algorithm_Guassian(y, op, c)
% Drop-in for SAPG/SAPG_algorithm_Guassian.m:7-308 - same signature, same `results` fields.
% The MYULA warm-up, the SAPG main loop and the traces run on the GPU (libsbd.so); the function
% handles in `op` are not called: the engine implements the model they encode from the plain
% fields the demo already stores (psf_size, phi, lambda, gamma, w1, w2, sigma*, ...).
P = sbd_pack(0, op, c);
X0 = []; if isfield(op, 'X0'), X0 = op.X0; end
noise = []; if isfield(op, 'noise'), noise = op.noise; end       % optional explicit randn stream
r = sbd_mex('sapg', double(y), X0, [], 0, op.psf_size, op.phi, P, noise);
theta_EB = r.EB(1); w1_EB = r.EB(2); w2_EB = r.EB(3); sigma_EB = r.EB(4);
results.logPiTrace_WU = r.logPiTrace_WU; results.execTimeFindParameters = r.seconds;
results.last_samp = r.last_samp; results.logPiTraceX = r.logPiTraceX; results.gXTrace = r.gXTrace;
results.theta_EB = theta_EB; results.last_theta = r.thetas(end); results.thetas = r.thetas;
results.mean_thetas = r.mean_theta(:); results.tol_thetas = r.tol_theta;
results.w1_EB = w1_EB; results.last_w1 = r.psi0(end); results.w1s = r.psi0;
results.mean_w1s = r.mean_psi0(:); results.tol_w1s = r.tol_psi0;
results.w2_EB = w2_EB; results.last_w2 = r.psi1(end); results.w2s = r.psi1;
results.mean_w2s = r.mean_psi1(:); results.tol_w2s = r.tol_psi1;
results.sigma_EB = sigma_EB; results.last_sigma = r.sigmas(end); results.sigmas = r.sigmas;
results.mean_sigmas = r.mean_sigma(:); results.tol_sigma = r.tol_sigma;
results.c_theta = c.theta; results.c_w1 = c.w1; results.c_w2 = c.w2; results.Xlast_sample = r.X_last;
results.c_sigma = c.sigma; results.err_psf = r.err_psf;
results.grad_theta = r.grad_theta; results.grad_w1 = r.grad_psi0; results.grad_w2 = r.grad_psi1;
results.grad_sigma = r.grad_sigma; results.options = op;
if isfield(r, 'posterior'), results = sbd_posterior(results, r); end   % only with op.post_levels > 0
end
