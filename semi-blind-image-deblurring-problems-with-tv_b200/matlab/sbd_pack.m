function [P, r2res] = sbd_pack(model, op, c)
% Flatten the reference's `op` (+ `c`) structs into the POD the C ABI takes (include/sbd.h: sbd_params).
if ~isfield(op, 'warmup'), op.warmup = 100; end                      % Guassian.m:19-21
P.samples = op.samples; P.warmup = op.warmup; P.burnIn = op.burnIn; P.n_chains = 1;
if isfield(op, 'n_chains'), P.n_chains = op.n_chains; end
switch model
    case 0
        names = {'w1', 'w2'};
        P.gam = c.gam * op.gamma; P.lamb = c.lam * op.lambda;        % Guassian.m:30-31
        P.c_theta = c.theta; P.c_sigma2 = c.sigma; P.c_psi = [c.w1 c.w2];
        P.sigma2_fixed = op.sigma_init; P.err_psf_lag = 1;           % Guassian.m:190, :203
    case 1
        names = {'alpha', 'beta'};
        P.gam = op.gamma; P.lamb = op.lambda;
        P.c_theta = 0.1; P.c_psi = [10 10000]; P.c_sigma2 = 10000;    % moffat.m:135-138
        P.sigma2_fixed = op.sigma^2; P.err_psf_lag = 0;              % moffat.m:197
    case 2
        names = {'b'};
        P.gam = op.gamma; P.lamb = op.lambda;
        P.c_theta = 0.01; P.c_psi = [100 0]; P.c_sigma2 = 10000;      % laplace.m:139-141
        P.sigma2_fixed = op.sigma^2; P.err_psf_lag = 0;              % laplace.m:182
end
P.prox_lambda = op.lambda;                                           % run_Gaussian_demo.m:191
% Chambolle options: the reference hard-wires them inside op.proxG (run_Gaussian_demo.m:188-191: 'maxiter',
% op.chambolleit with the defaults tol = 1e-3, tau = 0.249 of chambolle_prox_TV_stop.m:77-78).  A handle cannot be
% inspected, so the plain fields are honoured instead (same names as the Python front end, host.make_params).
P.chambolle_maxiter = 25; P.chambolle_tol = 1e-3; P.chambolle_tau = 0.249;
if isfield(op, 'chambolleit'), P.chambolle_maxiter = op.chambolleit; end
if isfield(op, 'chambolle_tol'), P.chambolle_tol = op.chambolle_tol; end
if isfield(op, 'chambolle_tau'), P.chambolle_tau = op.chambolle_tau; end
% The closures in op (proxG, gradF, logPi, f, g, grad_*) are NOT called: the engine implements the model they
% encode.  Say so once, so that an edited closure does not silently go unused.
hnames = {'proxG', 'gradF', 'logPi', 'f', 'g', 'gradF_sigma'};
for k = 1:numel(hnames)
    if isfield(op, hnames{k}) && ~(isfield(op, 'sbd_quiet') && op.sbd_quiet)
        warning('sbd:handlesIgnored', ['op.' hnames{k} ' (and the other function handles in op) are not called by the ' ...
                'GPU engine; set op.chambolleit / op.chambolle_tol / op.chambolle_tau or op.sbd_quiet = 1']);
        break;
    end
end
P.th_init = op.th_init; P.min_th = op.min_th; P.max_th = op.max_th;
P.psi_init = [0 0]; P.psi_min = [0 0]; P.psi_max = [0 0]; P.psi_fixed = [0 0]; P.psi_true = [0 0]; P.fix_psi = [0 0];
for k = 1:numel(names)
    n = names{k};
    P.psi_init(k) = op.([n '_init']); P.psi_min(k) = op.(['min_' n]); P.psi_max(k) = op.(['max_' n]);
    P.psi_fixed(k) = op.(n); P.psi_true(k) = op.(n); P.fix_psi(k) = op.(['fix_' n]);
end
P.sigma2_init = op.sigma_init; P.sigma2_min = op.sigma_min; P.sigma2_max = op.sigma_max; P.fix_sigma = op.fix_sigma;
P.d_scale = op.d_scale; P.d_exp = op.d_exp; P.seed = 1;
if isfield(op, 'seed'), P.seed = op.seed; end
P.use_graph = -1;                                                    % automatic: CUDA-graph replay for small images
if isfield(op, 'use_graph'), P.use_graph = op.use_graph; end
if isfield(op, 'post_levels'), P.post_levels = op.post_levels; end   % posterior statistics (sbd_posterior.m)
if isfield(op, 'post_batch'), P.post_batch = op.post_batch; end      % their ESS / MCSE / split Rhat (-1: auto)
r2res = names;
end
