function [T, rmse, n_used, status, best, idx] = pcreg_icp_windows(model, src, T0, opts, w_src)
%% pcreg_icp_windows -- pcreg_icp for a whole batch of matching windows in ONE GPU call, each window's poses against its own
% source cloud.  Replaces the per-window ICP polish of slideMatchingWindow_v2.m:178-198 / completeExperiment.m:265:
%     parfor w = 1:W, [T{w}, rmse{w}, ...] = pcreg_icp(model, src{w}, T0{w}, opts); end
% model: pcreg_mex('model_create', ...) handle; src: 1xW cell of N_w x 3 source clouds; T0: 1xW cell of 4x4xH_w initial poses
% (H_w may be 0); opts as for pcreg_icp; w_src (optional): 1xW cell of N_w x 1 weights.
% Outputs: 1xW cells T (4x4xH_w), rmse, n_used, status (H_w x 1), idx (N_w x H_w, 1-based), and best (W x 1, 1-based within the
% window, 0 where the window has no hypothesis).  Each window's outputs are what pcreg_icp returns for that window alone.
    W = numel(src);
    ns = cellfun(@(p) size(p, 1), src(:));
    H = cellfun(@(t) size(t, 3) * (numel(t) > 0), T0(:));
    soff = [0; cumsum(ns)];
    hoff = [0; cumsum(H)];
    T0all = zeros(16, hoff(end));
    for w = 1:W
        T0all(:, hoff(w) + 1 : hoff(w + 1)) = reshape(double(T0{w}), 16, H(w));
    end
    args = {model, double(vertcat(src{:})), soff, T0all, hoff, opts};
    if nargin > 4, args{end + 1} = double(vertcat(w_src{:})); end
    [T16, r, nu, st, best, idx16] = pcreg_mex_windows(args{:});
    T = cell(1, W); rmse = cell(1, W); n_used = cell(1, W); status = cell(1, W); idx = cell(1, W);
    ioff = [0; cumsum(H .* ns)];
    for w = 1:W
        h = hoff(w) + 1 : hoff(w + 1);
        T{w} = reshape(T16(:, h), 4, 4, H(w));
        rmse{w} = r(h); n_used{w} = nu(h); status{w} = st(h);
        idx{w} = reshape(idx16(ioff(w) + 1 : ioff(w + 1)), ns(w), H(w));
    end
end
