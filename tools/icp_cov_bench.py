"""What the pose covariance pass (include/pcreg.h: pcreg_icp_covariance) costs on the C3 and C4 workloads of bench.py, how well it is
calibrated, and what it says about the C3 winner.

    python tools/icp_cov_bench.py [--steps 3] [--c4-hyp 100000] [--out profiles/r11_icp_cov.json]

Cost: per workload, the workload's ICP call (pcreg_icp_batch_dev) and the covariance pass at that call's final poses
(pcreg_icp_covariance_dev, same options, ref = the patch centre, one target) are timed ALTERNATELY in one process, each step with
bench.py's L2 flush before it, outside the CUDA-event bracket; median, min and max of the steps.
C3 winner: its predicted TRE at the patch centre (the image of the source centroid) against its actual distance there from T_gt.
Calibration: 64 draws of sigma = 0.3 mm noise on one 2000-point patch of a 300 000-point model, each its own window, ICP from T_gt
(point-to-point PLAIN 60 iterations, point-to-plane PLAIN 20), then the covariance at the final poses: empirical / predicted std along
the principal directions of the mean predicted covariance (tests/icp_cov_reference.py).  The card name and power limit are read in
the same run.  Needs a GPU; there is no CPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402  (workload definitions, L2 flush, timing brackets)
from icp_extrap_bench import c3_inputs, c4_inputs  # noqa: E402
from icp_stop_bench import card  # noqa: E402


def run_workload(P, torch, w, model, src, T0, w_src, T_gt, mkw, steps, warmup):
    from pcreg_b200 import torch_ops
    dev = torch.device("cuda", 0)
    m = P.Model(model, grid=True)
    m.compute_normals(6)
    mode = dict(plain=P.ICP_PLAIN, knn=P.ICP_KNN, weighted=P.ICP_WEIGHTED)[mkw["mode"]]
    H, ns = T0.shape[0], src.shape[0]
    src_cm = torch_ops.src_to_abi_t(torch.from_numpy(np.asarray(src)).to(dev))
    T0_abi = torch_ops.T_to_abi_t(torch.from_numpy(T0).to(dev))
    w_t = torch.from_numpy(w_src).to(dev) if w_src is not None else None
    flush = bench.Flusher(torch, dev)
    opts = P.icp_opts(mode=mode, iters=w["iters"], k_frac=0.85, R_w=3.5, thDist2=mkw["thDist2"], nn=P.NN_GRID)
    icp_out = torch_ops.IcpDeviceBuffers(H, ns, w["iters"], dev)
    cov_out = torch_ops.IcpCovDeviceBuffers(H, 1, dev)
    csrc = np.asarray(src, dtype=np.float64).mean(axis=0)
    centre = csrc @ T_gt[:3, :3] + T_gt[3, :3]

    def icp():
        torch_ops.icp_batch_device(m, src_cm, w_t, T0_abi, opts, icp_out)

    def cov():
        torch_ops.icp_covariance_device(m, src_cm, [0, ns], w_t, icp_out.T, [0, H], opts, cov_out, ref=centre, targets=[centre])

    steps_by = dict(icp=icp, cov=cov)
    for _ in range(warmup):
        icp(); cov()
    torch.cuda.synchronize()
    times = {k: [] for k in steps_by}
    for _ in range(steps):                                        # alternate: one step of each per round
        for k, f in steps_by.items():
            times[k] += bench.time_steps(torch, f, 1, flush, torch.cuda.synchronize)
    T = torch_ops.T_from_abi_t(icp_out.T).cpu().numpy()
    rmse = icp_out.rmse.cpu().numpy()
    best = int(np.nanargmin(rmse))
    tre = cov_out.tre.cpu().numpy()[:, 0]
    status = cov_out.status.cpu().numpy()
    Tb = T[best]
    res = dict(workload=w["desc"], hypotheses=H, source_points=ns, model_points=w["nm"], icp_iters=w["iters"])
    for k in steps_by:
        ms = np.asarray(times[k])
        res[k] = dict(ms_per_step=float(np.median(ms)), ms_min=float(ms.min()), ms_max=float(ms.max()), ms_all=ms.tolist())
    res["cov_over_icp"] = res["cov"]["ms_per_step"] / res["icp"]["ms_per_step"]
    res["cov_status_1_share"] = float((status == 1).mean())
    res["winner"] = dict(index=best, rmse=float(rmse[best]), status=int(status[best]), predicted_tre_mm=float(tre[best]),
                         sigma2=float(cov_out.sigma2[best].item()),
                         actual_centre_error_mm=float(np.linalg.norm((csrc @ Tb[:3, :3] + Tb[3, :3]) - centre)),
                         cov=cov_out.cov[best].cpu().numpy().reshape(6, 6).tolist())
    m.destroy()
    return res


def calibration(P, draws=64, sigma=0.3):
    from icp_cov_reference import calibration_ratios, pose_error
    from pcreg_b200 import synth
    model = synth.make_model(300_000, 7)
    m = P.Model(model, grid=True)
    m.compute_normals(10)
    clean, T_gt, c = synth.make_source(model, 2000, 0.0, 11)
    Ti = np.linalg.inv(T_gt)
    g = synth.rng(12)
    srcs = [clean + g.normal(0.0, sigma, clean.shape) for _ in range(draws)]
    out = {}
    for metric, iters in (("point_to_point", 60), ("point_to_plane", 20)):
        icp = P.icp_batch_windows(m, srcs, [T_gt[None]] * draws, mode=P.ICP_PLAIN, iters=iters, nn=P.NN_GRID, metric=metric)
        Ts = [r["T"][0] for r in icp]
        cov = P.icp_covariance_windows(m, srcs, [t[None] for t in Ts], mode=P.ICP_PLAIN, nn=P.NN_GRID, ref=c, targets=[c])
        ratio, pred = calibration_ratios(np.stack([r["cov"][0] for r in cov]), [pose_error(t, T_gt, c) for t in Ts])
        s_c = c @ Ti[:3, :3] + Ti[3, :3]                          # the source point T_gt puts at the patch centre
        err_c = np.array([np.linalg.norm(s_c @ t[:3, :3] + t[3, :3] - c) for t in Ts])
        out[metric] = dict(iters=iters, predicted_std=pred.tolist(), empirical_over_predicted=ratio.tolist(),
                           predicted_rms_tre_centre_mm=float(np.sqrt(np.mean([r["tre"][0][0] ** 2 for r in cov]))),
                           empirical_rms_centre_error_mm=float(np.sqrt(np.mean(err_c ** 2))),
                           sigma2_mean=float(np.mean([r["sigma2"][0] for r in cov])), status_1=int(sum(r["status"][0] for r in cov)))
    m.destroy()
    return dict(draws=draws, sigma_mm=sigma, model_points=300_000, source_points=2000, ref="patch centre", metrics=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--c4-hyp", type=int, default=bench.C4["hyp"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_icp_cov.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("icp_cov_bench.py: no CUDA device (there is no CPU path)")
    import pcreg_b200 as P
    P.init(0)
    out = dict(card=card(), steps=args.steps, warmup=args.warmup,
               l2="flushed: %d MB written before every timed step, outside its CUDA-event bracket" % (bench.L2_FLUSH_BYTES >> 20),
               schedule="ICP call and covariance pass alternated within each round; median of the steps", workloads={})
    out["calibration"] = calibration(P)
    print(json.dumps(out["calibration"]), flush=True)
    out["workloads"]["c3"] = run_workload(P, torch, *c3_inputs(), args.steps, args.warmup)
    print(json.dumps(out["workloads"]["c3"]), flush=True)
    out["workloads"]["c4_polish"] = run_workload(P, torch, *c4_inputs(args.c4_hyp), args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
