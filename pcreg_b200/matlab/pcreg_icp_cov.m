function [cov, sigma2, rmse, n_used, status, tre, info] = pcreg_icp_cov(model, src, T, opts, ref, targets, w_src)
%% pcreg_icp_cov -- pose covariance and predicted target registration error of given poses (include/pcreg.h: pcreg_icp_covariance).
% One scoring pass per pose with pcreg_icp's correspondences, rejection, mode and weights (opts as for pcreg_icp; iters is ignored),
% no update; the model needs normals.  Typically T is what pcreg_icp / pcreg_icp_windows returned.
% model: pcreg_mex('model_create', ...) handle; src: N x 3 source cloud, or a 1xW cell of them with T a 1xW cell of 4x4xH_w poses;
% ref (optional, [] = origin): the model-frame point the rotation is about; targets (optional): K x 3 model-frame points;
% w_src (optional): N x 1 weights (a cell per window with a cell src).
% Outputs per pose (cells per window with a cell src): cov (6x6xH, unknowns [omega; tau], rad and model units), sigma2, rmse,
% n_used, status (1: degenerate, cov and tre NaN), tre (H x K, predicted RMS displacement of each target), info (6x6xH, the
% unscaled Hessian; its small-eigenvalue eigenvectors are the motions the patch leaves free).
    if nargin < 5, ref = []; end
    if nargin < 6, targets = []; end
    if nargin < 7, w_src = []; end
    cells = iscell(src);
    if ~cells, src = {src}; T = {T}; if ~isempty(w_src), w_src = {w_src}; end, end
    W = numel(src);
    ns = cellfun(@(p) size(p, 1), src(:));
    H = cellfun(@(t) size(t, 3) * (numel(t) > 0), T(:));
    soff = [0; cumsum(ns)];
    hoff = [0; cumsum(H)];
    Tall = zeros(16, hoff(end));
    for w = 1:W
        Tall(:, hoff(w) + 1 : hoff(w + 1)) = reshape(double(T{w}), 16, H(w));
    end
    w_all = [];
    if ~isempty(w_src), w_all = double(vertcat(w_src{:})); end
    [c36, s2, r, nu, st, tr, i36] = pcreg_mex_cov(model, double(vertcat(src{:})), soff, Tall, hoff, opts, double(ref), double(targets), w_all);
    cov = cell(1, W); sigma2 = cell(1, W); rmse = cell(1, W); n_used = cell(1, W); status = cell(1, W); tre = cell(1, W); info = cell(1, W);
    for w = 1:W
        h = hoff(w) + 1 : hoff(w + 1);
        cov{w} = reshape(c36(:, h), 6, 6, H(w)); info{w} = reshape(i36(:, h), 6, 6, H(w));
        sigma2{w} = s2(h); rmse{w} = r(h); n_used{w} = nu(h); status{w} = st(h); tre{w} = tr(h, :);
    end
    if ~cells
        cov = cov{1}; sigma2 = sigma2{1}; rmse = rmse{1}; n_used = n_used{1}; status = status{1}; tre = tre{1}; info = info{1};
    end
end
