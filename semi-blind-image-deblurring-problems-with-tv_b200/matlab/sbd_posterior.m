function results = sbd_posterior(results, r)
% Posterior statistics of a run with op.post_levels = L > 0 (include/sbd.h sbd_posterior_stats, DESIGN.md
% "Posterior statistics").  sbd_mex('sapg', ...) returns them as r.posterior, one field per block size (s1, s2, s4,
% ...); this sets
%   results.posterior     struct array, one element per block size 1, 2, ..., 2^(L-1), with fields
%                         scale, n, chains, mean, within, between, var, std, Rhat
%   results.posteriorvar, results.posteriorstd, results.Rhat      the pixel-scale (s = 1) var, std and Rhat
% and, with op.post_batch (sbd_posterior_diagnostics), the struct array also has the fields batch_mean, batch_within,
% batch_between, half_mean, half_within, half_between, batch_len, n_batches, half_n, ESS, MCSE, Rhat_split, and
%   results.ESS, results.MCSE, results.Rhat_split                 their pixel-scale (s = 1) values
% and, with op.post_ci = alpha (sbd_posterior_quantiles), the fields ci_alpha, ci_count, lower, median, upper,
% ci_width (the 1 - alpha credible interval and the posterior median), and
%   results.posteriormedian, results.CI_lower, results.CI_upper   their pixel-scale (s = 1) values
f = fieldnames(r.posterior);
for k = 1:numel(f)
    post(k) = r.posterior.(f{k});
end
results.posterior = post;
results.posteriorvar = post(1).var; results.posteriorstd = post(1).std; results.Rhat = post(1).Rhat;
if isfield(post, 'ESS')
    results.ESS = post(1).ESS; results.MCSE = post(1).MCSE; results.Rhat_split = post(1).Rhat_split;
end
if isfield(post, 'median')
    results.posteriormedian = post(1).median; results.CI_lower = post(1).lower; results.CI_upper = post(1).upper;
end
end
