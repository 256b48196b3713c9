"""What the point-to-plane ICP metric (include/pcreg.h: pcreg_icp_batch_metric) buys on the C3 and C4 workloads of bench.py, and
what the device normals (pcreg_model_compute_normals) cost on the C3, C4 and C5 models.

    python tools/icp_plane_bench.py [--steps 3] [--c4-hyp 100000] [--out profiles/r04_icp_plane.json]

Normals: compute_normals(k=6) on each model, one untimed call then `--steps` timed calls (host clock around the synchronous call).
ICP: for each workload the settings (point-to-point at the workload's iteration count, point-to-plane at several counts) are timed
ALTERNATELY in one process (round r times every setting once), each step through the device entry (pcreg_icp_batch_metric_dev)
with bench.py's 256 MB L2 flush before it, outside the CUDA-event bracket.  Reported per setting: ms per step (median, min, max),
hypotheses/s, the winner's distance from T_gt (translation, model units = mm; rotation, Frobenius norm of R - R_gt), the best
rmse, and the share of hypotheses that meet the reference's success criterion ||R R_gt' - I||_F < 0.5 (visualizeGTMatches.m:221,
417-421) together with a 0.1 mm translation bound.  The card name and power limit are read in the same run.  Needs a GPU; there is
no CPU path.
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
from icp_stop_bench import c3_inputs, c4_inputs, card  # noqa: E402

C3_SETTINGS = [("p2p_30", "point_to_point", 30)] + [("plane_%d" % k, "point_to_plane", k) for k in (5, 8, 10, 15, 30)]
C4_SETTINGS = [("p2p_20", "point_to_point", 20)] + [("plane_%d" % k, "point_to_plane", k) for k in (5, 10, 20)]


def normals_time(P, model, steps):
    m = P.Model(model, grid=True)
    m.compute_normals(6)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        m.compute_normals(6)                                     # returns after the kernel and the copies have finished
        ts.append((time.perf_counter() - t0) * 1e3)
    m.destroy()
    return dict(model_points=int(np.asarray(model).shape[0]), k=6, ms=float(np.median(ts)), ms_all=ts)


def pose_errors(T, T_gt):
    R, Rg = T[:, :3, :3], T_gt[:3, :3]
    rot_fro = np.linalg.norm(R - Rg, axis=(1, 2))
    rel = np.linalg.norm(R @ Rg.T - np.eye(3), axis=(1, 2))
    trans = np.linalg.norm(T[:, 3, :3] - T_gt[3, :3], axis=1)
    return rot_fro, rel, trans


def run_workload(P, torch, w, model, src, T0, w_src, mkw, T_gt, settings, steps, warmup):
    from pcreg_b200 import torch_ops
    dev = torch.device("cuda", 0)
    m = P.Model(model, grid=True)
    m.compute_normals(6)
    mode = dict(plain=P.ICP_PLAIN, knn=P.ICP_KNN, weighted=P.ICP_WEIGHTED)[mkw["mode"]]
    H, ns = T0.shape[0], src.shape[0]
    src_cm = torch_ops.src_to_abi_t(torch.from_numpy(src).to(dev))
    T0_abi = torch_ops.T_to_abi_t(torch.from_numpy(T0).to(dev))
    w_t = torch.from_numpy(w_src).to(dev) if w_src is not None else None
    flush = bench.Flusher(torch, dev)
    opts = {s: P.icp_opts(mode=mode, iters=it, k_frac=0.85, R_w=3.5, thDist2=mkw["thDist2"], nn=P.NN_GRID) for s, _, it in settings}
    bufs = {s: torch_ops.IcpDeviceBuffers(H, ns, it, dev) for s, _, it in settings}

    def step(s, metric):
        torch_ops.icp_batch_device(m, src_cm, w_t, T0_abi, opts[s], bufs[s], metric=metric)

    for _ in range(warmup):
        for s, metric, _ in settings:
            step(s, metric)
    torch.cuda.synchronize()
    times = {s: [] for s, _, _ in settings}
    for _ in range(steps):                                        # alternate: one step of every setting per round
        for s, metric, _ in settings:
            times[s] += bench.time_steps(torch, lambda: step(s, metric), 1, flush, torch.cuda.synchronize)
    res = {}
    for s, metric, it in settings:
        b = bufs[s]
        T = torch_ops.T_from_abi_t(b.T).cpu().numpy()
        rmse = b.rmse.cpu().numpy()
        best = int(b.best.item())
        ms = np.asarray(times[s])
        rot_fro, rel, trans = pose_errors(T, T_gt)
        res[s] = dict(metric=metric, iters=it, ms_per_step=float(np.median(ms)), ms_min=float(ms.min()), ms_max=float(ms.max()),
                      ms_all=ms.tolist(), hyp_per_s=H / (float(np.median(ms)) * 1e-3), best=best, best_rmse=float(rmse[best]),
                      winner_vs_gt=dict(trans_mm=float(trans[best]), rot_fro=float(rot_fro[best])),
                      success_frac=float(np.mean((rel < 0.5) & (trans < 0.1))),
                      degenerate_frac=float(np.mean(b.status.cpu().numpy() != 0)))
    m.destroy()
    return dict(workload=w["desc"], hypotheses=H, source_points=ns, model_points=w["nm"], settings=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--c4-hyp", type=int, default=bench.C4["hyp"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_icp_plane.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("icp_plane_bench.py: no CUDA device (there is no CPU path)")
    import pcreg_b200 as P
    from pcreg_b200 import synth
    P.init(0)
    out = dict(card=card(), steps=args.steps, warmup=args.warmup,
               l2="flushed: %d MB written before every timed ICP step, outside its CUDA-event bracket" % (bench.L2_FLUSH_BYTES >> 20),
               schedule="settings alternated within each round", normals={}, workloads={})
    w3, model3, src3, T03, ws3, mkw3 = c3_inputs()
    T_gt3 = bench.make_inputs(w3, 0)[4]
    c5 = bench.WORKLOADS["c5"]
    for name, model in (("c3", model3), ("c4", synth.make_model(bench.C4["nm"], bench.C4["seed"])),
                        ("c5", synth.make_model(c5["nm"], c5["seed"]))):
        out["normals"][name] = normals_time(P, model, args.steps)
        print(name, json.dumps(out["normals"][name]), flush=True)
    out["workloads"]["c3"] = run_workload(P, torch, w3, model3, src3, T03, ws3, mkw3, T_gt3, C3_SETTINGS, args.steps, args.warmup)
    print(json.dumps(out["workloads"]["c3"]["settings"]), flush=True)
    w4, model4, src4, T04, ws4, mkw4 = c4_inputs(args.c4_hyp)
    c = bench.C4
    T_gt4 = synth.make_source(model4, c["ns"], 0.3, c["seed"])[1]
    out["workloads"]["c4_polish"] = run_workload(P, torch, w4, model4, src4, T04, ws4, mkw4, T_gt4, C4_SETTINGS, args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
