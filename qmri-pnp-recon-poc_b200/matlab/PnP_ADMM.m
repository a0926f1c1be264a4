function [x, info] = PnP_ADMM(y, param)
% Drop-in for main_files/algorithms/PnP_ADMM/PnP_ADMM.m (same signature and param fields:
% iter, gamma, cg_tol, F, gt_tsmi, X0, net, denoiser_type, noise_map).
% [x, info] = PnP_ADMM(y, param) also returns the per-iteration progress the reference prints (PnP_ADMM.m:106-109), recorded on
% the GPU inside the loop: info.dc_res = norm(y - F.forward(x_k)) / norm(y) and info.gt_err = norm(param.gt_tsmi - x_k) /
% norm(param.gt_tsmi), iter x S doubles (x_k: the x-update of iteration k, before the denoiser; gt_err is [] without gt_tsmi).
% param.net is either a handle returned by qmri_unetres_load (whole loop on the GPU) or any function handle @(v)
% (pluggable prox, host hop).  param.F: the struct from qmri_fft_operator (carries the operator handle), or the reference's
% own closures over P.for / P.adj (main_recon_tsmis_FFT.m:228-229) - then the operator built last by setup_subsampling_* is
% used, after checking on a probe image that param.F.forward really is that operator.
if ~isfield(param, 'denoiser_type'), param.denoiser_type = 'single_level'; end
if isfield(param.F, 'handle')
    h = param.F.handle;
else
    h = qmri_b200_mex('last_op');
    if h == 0, error('qmri:param', 'param.F carries no operator handle and no operator has been built'); end
    probe = randn(size(param.X0));
    ya = param.F.forward(probe); yb = qmri_b200_mex('forward', h, probe);
    if numel(ya) ~= numel(yb) || norm(ya(:) - yb(:)) > 1e-4 * norm(yb(:))
        error('qmri:param', 'param.F is not the operator built by the last setup_subsampling_* call; build F with qmri_fft_operator(P)');
    end
end
if nargout >= 2
    [x, info] = qmri_b200_mex('pnp_admm', h, double(y), param);
else
    x = qmri_b200_mex('pnp_admm', h, double(y), param);
end
end
