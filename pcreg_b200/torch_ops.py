"""Device-resident entry points: torch is only the plumbing (device memory, streams,
torch.distributed); the compute is libpcreg_b200.so through pcreg_icp_batch_dev."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L
from .api import GICP_EPS, ICP_PLANE_TO_PLANE, METRICS, PLANE_TO_PLANE, Model, icp_opts


def T_to_abi_t(T: torch.Tensor) -> torch.Tensor:
    """[H,4,4] math layout -> contiguous MATLAB column-major 16-double records."""
    return T.transpose(-1, -2).contiguous()


def T_from_abi_t(buf: torch.Tensor) -> torch.Tensor:
    return buf.view(-1, 4, 4).transpose(-1, -2).contiguous()


def src_to_abi_t(src: torch.Tensor) -> torch.Tensor:
    """[ns,3] -> column-major float64 (x[ns], y[ns], z[ns]) on the same device."""
    return src.to(torch.float64).t().contiguous()


class IcpDeviceBuffers:
    """Output tensors of one batched ICP call, allocated once and reused across steps."""

    def __init__(self, nhyp: int, ns: int, iters: int, device, want_idx=False, want_hist=False, want_n_iter=False, want_n_extrap=False):
        f64, i32 = torch.float64, torch.int32
        self.T = torch.empty((nhyp, 16), dtype=f64, device=device)
        self.rmse = torch.empty(nhyp, dtype=f64, device=device)
        self.n_used = torch.empty(nhyp, dtype=i32, device=device)
        self.status = torch.empty(nhyp, dtype=i32, device=device)
        self.idx = torch.empty((nhyp, ns), dtype=i32, device=device) if want_idx else None
        self.hist = torch.empty((nhyp, iters + 1), dtype=f64, device=device) if want_hist else None
        self.best = torch.empty(1, dtype=torch.int64, device=device)
        # filled by a call with a tolerance stop: pose updates applied, 1 = stopped by the tolerance
        self.n_iter = torch.empty(nhyp, dtype=i32, device=device) if want_n_iter else None
        self.converged = torch.empty(nhyp, dtype=i32, device=device) if want_n_iter else None
        # filled by a call with extrapolation: updates that extrapolated
        self.n_extrap = torch.empty(nhyp, dtype=i32, device=device) if want_n_extrap else None


class IcpWindowsDeviceBuffers(IcpDeviceBuffers):
    """Output tensors of one windowed call (icp_windows_device): per-hypothesis outputs as IcpDeviceBuffers, idx ragged (n_idx =
    sum over the windows of H_w * ns_w, window-major) and best [nwin]."""

    def __init__(self, nhyp: int, n_idx: int, nwin: int, iters: int, device, want_idx=False, want_hist=False, want_n_iter=False,
                 want_n_extrap=False):
        super().__init__(nhyp, 0, iters, device, False, want_hist, want_n_iter, want_n_extrap)
        self.idx = torch.empty(n_idx, dtype=torch.int32, device=device) if want_idx else None
        self.best = torch.empty(nwin, dtype=torch.int64, device=device)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _extrap_dev(model, src_cm, soff, w_src, hoff, T0_abi, opts, out, st, stop, extrap):
    L.check(L.lib().pcreg_icp_batch_extrap_dev(model.handle, _p(src_cm), soff.ctypes.data_as(L.c_i64p), _p(w_src), hoff.ctypes.data_as(L.c_i64p),
                                               soff.shape[0] - 1, _p(T0_abi), C.byref(opts), C.byref(stop) if stop is not None else None,
                                               C.byref(extrap), _p(out.T), _p(out.rmse), _p(out.n_used), _p(out.status), _p(out.idx),
                                               _p(out.hist), _p(out.best), _p(out.n_iter), _p(out.converged), _p(out.n_extrap),
                                               C.c_void_p(st.cuda_stream)),
            "pcreg_icp_batch_extrap_dev")


def icp_batch_device(model: Model, src_cm: torch.Tensor, w_src, T0_abi: torch.Tensor, opts, out: IcpDeviceBuffers,
                     stream=None, stop=None, metric="point_to_point", src_normals=None, gicp_eps=GICP_EPS, extrap=None):
    """Run pcreg_icp_batch_dev on tensors already resident on the library's device.

    src_cm: float64 [3, ns] (column-major ns x 3); T0_abi: float64 [H,16] column-major records.
    stop: an api.icp_stop(tol_t, tol_r_deg, window) -> pcreg_icp_batch_stop_dev (out.n_iter / out.converged, when allocated,
    receive the stop outputs).  metric="point_to_plane" -> pcreg_icp_batch_metric_dev (needs model normals).
    metric="plane_to_plane" -> pcreg_icp_batch_gicp_dev: needs model normals and src_normals, a CUDA float64 [ns, 3] tensor.
    extrap: an api.icp_extrap(angle_deg, vmax_scale) -> pcreg_icp_batch_extrap_dev with one window (point-to-point only; out.n_extrap,
    when allocated, receives the updates that extrapolated)."""
    if not (src_cm.is_cuda and T0_abi.is_cuda):
        raise L.PcregError("icp_batch_device needs CUDA tensors (there is no CPU fallback)")
    assert src_cm.dtype == torch.float64 and src_cm.is_contiguous() and src_cm.shape[0] == 3
    assert T0_abi.dtype == torch.float64 and T0_abi.is_contiguous()
    ns = src_cm.shape[1]
    nhyp = T0_abi.shape[0]
    st = stream if stream is not None else torch.cuda.current_stream()
    if extrap is not None:
        if metric != "point_to_point":
            raise ValueError("extrap is defined for metric='point_to_point' only")
        _extrap_dev(model, src_cm, np.array([0, ns], dtype=np.int64), w_src, np.array([0, nhyp], dtype=np.int64), T0_abi, opts, out, st,
                    stop, extrap)
    elif metric == PLANE_TO_PLANE:
        if src_normals is None:
            raise ValueError("metric='plane_to_plane' needs src_normals (a CUDA float64 [ns, 3] tensor)")
        if not (src_normals.is_cuda and src_normals.dtype == torch.float64 and tuple(src_normals.shape) == (ns, 3)):
            raise ValueError("src_normals must be a CUDA float64 [ns, 3] tensor")
        sn_cm = src_normals.t().contiguous()                   # column-major ns x 3, ld = ns
        L.check(L.lib().pcreg_icp_batch_gicp_dev(model.handle, _p(src_cm), ns, _p(w_src), _p(sn_cm), float(gicp_eps), _p(T0_abi), nhyp,
                                                 C.byref(opts), C.byref(stop) if stop is not None else None, _p(out.T),
                                                 _p(out.rmse), _p(out.n_used), _p(out.status), _p(out.idx), _p(out.hist),
                                                 _p(out.best), _p(out.n_iter), _p(out.converged), C.c_void_p(st.cuda_stream)),
                "pcreg_icp_batch_gicp_dev")
    elif metric != "point_to_point":
        L.check(L.lib().pcreg_icp_batch_metric_dev(model.handle, _p(src_cm), ns, _p(w_src), _p(T0_abi), nhyp, C.byref(opts),
                                                   METRICS[metric], C.byref(stop) if stop is not None else None, _p(out.T),
                                                   _p(out.rmse), _p(out.n_used), _p(out.status), _p(out.idx), _p(out.hist),
                                                   _p(out.best), _p(out.n_iter), _p(out.converged), C.c_void_p(st.cuda_stream)),
                "pcreg_icp_batch_metric_dev")
    elif stop is None:
        L.check(L.lib().pcreg_icp_batch_dev(model.handle, _p(src_cm), ns, _p(w_src), _p(T0_abi), nhyp, C.byref(opts),
                                            _p(out.T), _p(out.rmse), _p(out.n_used), _p(out.status), _p(out.idx),
                                            _p(out.hist), _p(out.best), C.c_void_p(st.cuda_stream)),
                "pcreg_icp_batch_dev")
    else:
        L.check(L.lib().pcreg_icp_batch_stop_dev(model.handle, _p(src_cm), ns, _p(w_src), _p(T0_abi), nhyp, C.byref(opts),
                                                 C.byref(stop), _p(out.T), _p(out.rmse), _p(out.n_used), _p(out.status),
                                                 _p(out.idx), _p(out.hist), _p(out.best), _p(out.n_iter), _p(out.converged),
                                                 C.c_void_p(st.cuda_stream)),
                "pcreg_icp_batch_stop_dev")
    return out


def icp_windows_device(model: Model, src_cm: torch.Tensor, src_offsets, w_src, T0_abi: torch.Tensor, hyp_offsets, opts,
                       out: IcpWindowsDeviceBuffers, stream=None, stop=None, metric="point_to_point", src_normals=None, gicp_eps=GICP_EPS,
                       extrap=None):
    """Run pcreg_icp_batch_windows_dev on tensors already resident on the library's device.

    src_cm: float64 [3, ns_total], the windows' sources one after the other (column-major ns_total x 3); src_offsets / hyp_offsets:
    HOST sequences of nwin + 1 row / hypothesis offsets; T0_abi: float64 [H,16] column-major records grouped by window; w_src: CUDA
    float64 [ns_total] or None.  metric="plane_to_plane" needs src_normals, a CUDA float64 [ns_total, 3] tensor.  extrap: as
    icp_batch_device (pcreg_icp_batch_extrap_dev)."""
    if not (src_cm.is_cuda and T0_abi.is_cuda):
        raise L.PcregError("icp_windows_device needs CUDA tensors (there is no CPU fallback)")
    assert src_cm.dtype == torch.float64 and src_cm.is_contiguous() and src_cm.shape[0] == 3
    assert T0_abi.dtype == torch.float64 and T0_abi.is_contiguous()
    soff = np.ascontiguousarray(np.asarray(src_offsets, dtype=np.int64))
    hoff = np.ascontiguousarray(np.asarray(hyp_offsets, dtype=np.int64))
    nwin = soff.shape[0] - 1
    if hoff.shape[0] != nwin + 1 or soff[-1] != src_cm.shape[1] or hoff[-1] != T0_abi.shape[0]:
        raise ValueError("src_offsets / hyp_offsets must be nwin + 1 offsets ending at ns_total / the number of poses")
    st = stream if stream is not None else torch.cuda.current_stream()
    if extrap is not None:
        if metric != "point_to_point":
            raise ValueError("extrap is defined for metric='point_to_point' only")
        _extrap_dev(model, src_cm, soff, w_src, hoff, T0_abi, opts, out, st, stop, extrap)
        return out
    sn_cm = None
    if metric == PLANE_TO_PLANE:
        if src_normals is None or not (src_normals.is_cuda and src_normals.dtype == torch.float64 and tuple(src_normals.shape) == (src_cm.shape[1], 3)):
            raise ValueError("metric='plane_to_plane' needs src_normals, a CUDA float64 [ns_total, 3] tensor")
        sn_cm = src_normals.t().contiguous()
    mcode = ICP_PLANE_TO_PLANE if metric == PLANE_TO_PLANE else METRICS[metric]
    L.check(L.lib().pcreg_icp_batch_windows_dev(model.handle, _p(src_cm), soff.ctypes.data_as(L.c_i64p), _p(w_src), _p(sn_cm),
                                                float(gicp_eps), hoff.ctypes.data_as(L.c_i64p), nwin, _p(T0_abi), C.byref(opts), mcode,
                                                C.byref(stop) if stop is not None else None, _p(out.T), _p(out.rmse), _p(out.n_used),
                                                _p(out.status), _p(out.idx), _p(out.hist), _p(out.best), _p(out.n_iter), _p(out.converged),
                                                C.c_void_p(st.cuda_stream)),
            "pcreg_icp_batch_windows_dev")
    return out


class IcpCovDeviceBuffers:
    """Output tensors of one icp_covariance_device call: cov / info [H,36] (row-major 6x6), sigma2, rmse, n_used, status [H] and
    tre [H,ntarget]."""

    def __init__(self, nhyp: int, ntarget: int, device, want_info=False):
        f64, i32 = torch.float64, torch.int32
        self.cov = torch.empty((nhyp, 36), dtype=f64, device=device)
        self.info = torch.empty((nhyp, 36), dtype=f64, device=device) if want_info else None
        self.sigma2 = torch.empty(nhyp, dtype=f64, device=device)
        self.rmse = torch.empty(nhyp, dtype=f64, device=device)
        self.n_used = torch.empty(nhyp, dtype=i32, device=device)
        self.status = torch.empty(nhyp, dtype=i32, device=device)
        self.tre = torch.empty((nhyp, ntarget), dtype=f64, device=device) if ntarget else None


def icp_covariance_device(model: Model, src_cm: torch.Tensor, src_offsets, w_src, T_abi: torch.Tensor, hyp_offsets, opts,
                          out: IcpCovDeviceBuffers, ref=None, targets=None, stream=None):
    """Run pcreg_icp_covariance_dev on tensors already resident on the library's device: the pose covariance at the poses T_abi (layout
    of icp_windows_device).  ref (3) and targets ([K,3], model frame) are host values; out.tre must hold K columns."""
    if not (src_cm.is_cuda and T_abi.is_cuda):
        raise L.PcregError("icp_covariance_device needs CUDA tensors (there is no CPU fallback)")
    assert src_cm.dtype == torch.float64 and src_cm.is_contiguous() and src_cm.shape[0] == 3
    assert T_abi.dtype == torch.float64 and T_abi.is_contiguous()
    soff = np.ascontiguousarray(np.asarray(src_offsets, dtype=np.int64))
    hoff = np.ascontiguousarray(np.asarray(hyp_offsets, dtype=np.int64))
    nwin = soff.shape[0] - 1
    if hoff.shape[0] != nwin + 1 or soff[-1] != src_cm.shape[1] or hoff[-1] != T_abi.shape[0]:
        raise ValueError("src_offsets / hyp_offsets must be nwin + 1 offsets ending at ns_total / the number of poses")
    tg = np.zeros((0, 3)) if targets is None else np.asarray(targets, dtype=np.float64).reshape(-1, 3)
    K = tg.shape[0]
    if K and (out.tre is None or tuple(out.tre.shape) != (T_abi.shape[0], K)):
        raise ValueError("out.tre must be [H, ntarget]")
    tg_cm = np.asfortranarray(tg) if K else None
    rf = None if ref is None else np.ascontiguousarray(np.asarray(ref, dtype=np.float64).reshape(3))
    st = stream if stream is not None else torch.cuda.current_stream()
    f64p = L.c_f64p
    L.check(L.lib().pcreg_icp_covariance_dev(model.handle, _p(src_cm), soff.ctypes.data_as(L.c_i64p), _p(w_src), hoff.ctypes.data_as(L.c_i64p),
                                             nwin, _p(T_abi), C.byref(opts), rf.ctypes.data_as(f64p) if rf is not None else None,
                                             tg_cm.ctypes.data_as(f64p) if K else None, K, _p(out.cov), _p(out.info), _p(out.sigma2),
                                             _p(out.rmse), _p(out.n_used), _p(out.status), _p(out.tre) if K else None,
                                             C.c_void_p(st.cuda_stream)),
            "pcreg_icp_covariance_dev")
    return out
