"""What the plane-to-plane ICP metric (include/pcreg.h: pcreg_icp_batch_gicp) buys on the C3 and C4 workloads of bench.py against
point-to-point and point-to-plane, and what the source normals (cloud_normals) cost.

    python tools/icp_gicp_bench.py [--steps 3] [--k-large 20] [--c4-hyp 100000] [--out profiles/r05_icp_gicp.json]

Source normals: cloud_normals(src, k) for k = 6 and k = --k-large on the C3 (5 000 points) and C4 (20 000 points) sources, one untimed
call then `--steps` timed calls (host clock around the synchronous call: this is per-call work the caller pays).
ICP: for each workload the settings (point-to-point and point-to-plane at the iteration counts of tools/icp_plane_bench.py's winners,
plane-to-plane at several counts with the source normals of each k) are timed ALTERNATELY in one process (round r times every setting
once), each step through the device entries (pcreg_icp_batch_dev / _metric_dev / _gicp_dev) with bench.py's 256 MB L2 flush before
it, outside the CUDA-event bracket.  eps = 1e-3.  The model normals are compute_normals(6), as in tools/icp_plane_bench.py.  Reported
per setting as there: ms per step (median, min, max), hypotheses/s, the winner's distance from T_gt, the best rmse and the share of
hypotheses within ||R R_gt' - I||_F < 0.5 and 0.1 mm.  The card name and power limit are read in the same run.  Needs a GPU; there
is no CPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (workload definitions, L2 flush, timing brackets)
# the plane bench's workloads, card query and pose errors, so that these rows compare with profiles/r04_icp_plane.json
from icp_plane_bench import c3_inputs, c4_inputs, card, pose_errors  # noqa: E402

EPS = 1e-3


def settings(p2p_iters, plane_iters, gicp_iters, ks):
    """(name, metric, iters, k of the source normals or None)"""
    out = [("p2p_%d" % p2p_iters, "point_to_point", p2p_iters, None), ("plane_%d" % plane_iters, "point_to_plane", plane_iters, None)]
    return out + [("gicp_%d_k%d" % (it, k), "plane_to_plane", it, k) for k in ks for it in gicp_iters]


def normals_time(P, src, k, steps):
    P.cloud_normals(src, k)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        P.cloud_normals(src, k)                                  # returns after the kernel and the copies have finished
        ts.append((time.perf_counter() - t0) * 1e3)
    return dict(source_points=int(src.shape[0]), k=k, ms=float(np.median(ts)), ms_all=ts)


def run_workload(P, torch, w, model, src, T0, w_src, mkw, T_gt, sets, steps, warmup):
    from pcreg_b200 import torch_ops
    dev = torch.device("cuda", 0)
    m = P.Model(model, grid=True)
    m.compute_normals(6)
    mode = dict(plain=P.ICP_PLAIN, knn=P.ICP_KNN, weighted=P.ICP_WEIGHTED)[mkw["mode"]]
    H, ns = T0.shape[0], src.shape[0]
    src_cm = torch_ops.src_to_abi_t(torch.from_numpy(src).to(dev))
    T0_abi = torch_ops.T_to_abi_t(torch.from_numpy(T0).to(dev))
    w_t = torch.from_numpy(w_src).to(dev) if w_src is not None else None
    sn = {k: torch.from_numpy(P.cloud_normals(src, k)).to(dev) for k in {k for _, _, _, k in sets if k is not None}}
    flush = bench.Flusher(torch, dev)
    opts = {s: P.icp_opts(mode=mode, iters=it, k_frac=0.85, R_w=3.5, thDist2=mkw["thDist2"], nn=P.NN_GRID) for s, _, it, _ in sets}
    bufs = {s: torch_ops.IcpDeviceBuffers(H, ns, it, dev) for s, _, it, _ in sets}

    def step(s, metric, k):
        kw = dict(src_normals=sn[k], gicp_eps=EPS) if k is not None else {}
        torch_ops.icp_batch_device(m, src_cm, w_t, T0_abi, opts[s], bufs[s], metric=metric, **kw)

    for _ in range(warmup):
        for s, metric, _, k in sets:
            step(s, metric, k)
    torch.cuda.synchronize()
    times = {s: [] for s, _, _, _ in sets}
    for _ in range(steps):                                        # alternate: one step of every setting per round
        for s, metric, _, k in sets:
            times[s] += bench.time_steps(torch, lambda: step(s, metric, k), 1, flush, torch.cuda.synchronize)
    res = {}
    for s, metric, it, k in sets:
        b = bufs[s]
        T = torch_ops.T_from_abi_t(b.T).cpu().numpy()
        rmse = b.rmse.cpu().numpy()
        best = int(b.best.item())
        ms = np.asarray(times[s])
        rot_fro, rel, trans = pose_errors(T, T_gt)
        res[s] = dict(metric=metric, iters=it, src_normals_k=k, ms_per_step=float(np.median(ms)), ms_min=float(ms.min()),
                      ms_max=float(ms.max()), ms_all=ms.tolist(), hyp_per_s=H / (float(np.median(ms)) * 1e-3), best=best,
                      best_rmse=float(rmse[best]), winner_vs_gt=dict(trans_mm=float(trans[best]), rot_fro=float(rot_fro[best])),
                      success_frac=float(np.mean((rel < 0.5) & (trans < 0.1))),
                      degenerate_frac=float(np.mean(b.status.cpu().numpy() != 0)))
        print(s, json.dumps({x: res[s][x] for x in ("ms_per_step", "best_rmse", "winner_vs_gt", "success_frac")}), flush=True)
    m.destroy()
    return dict(workload=w["desc"], hypotheses=H, source_points=ns, model_points=w["nm"], eps=EPS, settings=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--k-large", type=int, default=20)
    ap.add_argument("--c4-hyp", type=int, default=bench.C4["hyp"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_icp_gicp.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("icp_gicp_bench.py: no CUDA device (there is no CPU path)")
    import pcreg_b200 as P
    from pcreg_b200 import synth
    P.init(0)
    ks = (6, args.k_large)
    out = dict(card=card(), steps=args.steps, warmup=args.warmup,
               l2="flushed: %d MB written before every timed ICP step, outside its CUDA-event bracket" % (bench.L2_FLUSH_BYTES >> 20),
               schedule="settings alternated within each round", cloud_normals={}, workloads={})
    w3, model3, src3, T03, ws3, mkw3 = c3_inputs()
    T_gt3 = bench.make_inputs(w3, 0)[4]
    w4, model4, src4, T04, ws4, mkw4 = c4_inputs(args.c4_hyp)
    c = bench.C4
    T_gt4 = synth.make_source(model4, c["ns"], 0.3, c["seed"])[1]
    for name, src in (("c3", src3), ("c4", src4)):
        for k in ks:
            out["cloud_normals"]["%s_k%d" % (name, k)] = r = normals_time(P, src, k, args.steps)
            print(name, json.dumps(r), flush=True)
    out["workloads"]["c3"] = run_workload(P, torch, w3, model3, src3, T03, ws3, mkw3, T_gt3,
                                          settings(30, 8, (5, 8, 10, 15, 30), ks), args.steps, args.warmup)
    out["workloads"]["c4_polish"] = run_workload(P, torch, w4, model4, src4, T04, ws4, mkw4, T_gt4,
                                                 settings(20, 10, (5, 10, 20), ks), args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
