"""What the ICP pose extrapolation (include/pcreg.h: pcreg_icp_extrap) buys on the C3 and C4 workloads of bench.py.

    python tools/icp_extrap_bench.py [--steps 3] [--c4-hyp 100000] [--out profiles/r08_icp_extrap.json]

For each workload the settings (iters 10 / 15 / 20 / 30 and the workload's iters with the default tolerance {0.01, 0.5, 3}, each
without and with extrapolation at its defaults {10, 25}; and the workload's iters with angle_deg = 1e-6, where the extrapolating
kernels run but almost nothing extrapolates: the cost of the mode itself) are timed ALTERNATELY in one process (round r times every setting once),
each step through the device entries (pcreg_icp_batch{,_stop}_dev without, pcreg_icp_batch_extrap_dev with) with bench.py's 256 MB
L2 flush before it, outside the CUDA-event bracket.  Reported per setting: ms per step (median, min, max), hypotheses/s, the best
rmse, the winner's distance from T_gt (translation of the source centroid's image in model units, ||R - R_gt||_F), the success share
(||R R_gt' - I||_F < 0.5, the reference's checkAlignment), the mean n_extrap and, with a tolerance, the mean n_iter.  The card name
and power limit are read in the same run.  Needs a GPU; there is no CPU path.
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

import bench  # noqa: E402  (workload definitions, L2 flush, timing brackets)
from icp_stop_bench import card  # noqa: E402

STOP = (0.01, 0.5, 3)
EX_DEFAULT, EX_ALMOST_OFF = (10.0, 25.0), (1e-6, 25.0)


def settings(iters):
    out = []
    for it in (10, 15, 20, 30):
        out += [("i%d" % it, it, None, None), ("i%d_ex" % it, it, None, EX_DEFAULT)]
    out += [("tol", iters, STOP, None), ("tol_ex", iters, STOP, EX_DEFAULT), ("i%d_ex_almost_off" % iters, iters, None, EX_ALMOST_OFF)]
    return out


def c3_inputs():
    w = bench.WORKLOADS["c3"]
    model, src, T0, w_src, T_gt = bench.make_inputs(w, 0)
    return w, model, src, T0, w_src, T_gt, dict(mode="knn", thDist2=0.0)


def c4_inputs(nhyp):
    from pcreg_b200 import synth
    c = bench.C4
    model = synth.make_model(c["nm"], c["seed"])
    src, T_gt, ctr = synth.make_source(model, c["ns"], 0.3, c["seed"])
    g = synth.rng(5)                                              # bench.c4_workload's seeds, first nhyp of them
    ang = np.deg2rad(g.uniform(0, 6, c["hyp"]))
    ax = g.standard_normal((c["hyp"], 3))
    tr = g.normal(0, 1.0, (c["hyp"], 3))
    T0 = np.stack([synth.perturb_pose(T_gt, ctr, synth.rot_axis_angle(ax[h], ang[h]), tr[h]) for h in range(nhyp)])
    w = dict(nm=c["nm"], ns=c["ns"], hyp=nhyp, iters=c["iters"], mode="plain", nn="grid", desc=c["desc"])
    return w, model, src, T0, None, T_gt, dict(mode="plain", thDist2=c["thDist2"])


def run_workload(P, torch, w, model, src, T0, w_src, T_gt, mkw, steps, warmup):
    from oracle.primitives import check_alignment
    from pcreg_b200 import torch_ops
    dev = torch.device("cuda", 0)
    m = P.Model(model, grid=True)
    mode = dict(plain=P.ICP_PLAIN, knn=P.ICP_KNN, weighted=P.ICP_WEIGHTED)[mkw["mode"]]
    H, ns = T0.shape[0], src.shape[0]
    src_cm = torch_ops.src_to_abi_t(torch.from_numpy(np.asarray(src)).to(dev))
    T0_abi = torch_ops.T_to_abi_t(torch.from_numpy(T0).to(dev))
    w_t = torch.from_numpy(w_src).to(dev) if w_src is not None else None
    flush = bench.Flusher(torch, dev)
    S = settings(w["iters"])
    opts = {s: P.icp_opts(mode=mode, iters=it, k_frac=0.85, R_w=3.5, thDist2=mkw["thDist2"], nn=P.NN_GRID) for s, it, _, _ in S}
    bufs = {s: torch_ops.IcpDeviceBuffers(H, ns, it, dev, want_n_iter=st is not None, want_n_extrap=ex is not None) for s, it, st, ex in S}
    stops = {s: (P.icp_stop(*st) if st is not None else None) for s, _, st, _ in S}
    extraps = {s: (P.icp_extrap(*ex) if ex is not None else None) for s, _, _, ex in S}

    def step(s):
        torch_ops.icp_batch_device(m, src_cm, w_t, T0_abi, opts[s], bufs[s], stop=stops[s], extrap=extraps[s])

    for _ in range(warmup):
        for s, *_ in S:
            step(s)
    torch.cuda.synchronize()
    times = {s: [] for s, *_ in S}
    for _ in range(steps):                                        # alternate: one step of every setting per round
        for s, *_ in S:
            times[s] += bench.time_steps(torch, lambda: step(s), 1, flush, torch.cuda.synchronize)
    c = np.asarray(src, dtype=np.float64).mean(axis=0)
    res = {}
    for s, it, st, ex in S:
        b = bufs[s]
        T = torch_ops.T_from_abi_t(b.T).cpu().numpy()
        rmse = b.rmse.cpu().numpy()
        best = int(b.best.item())
        ms = np.asarray(times[s])
        Tb = T[best]
        ok = np.array([check_alignment(T[h][:3, :3], T_gt[:3, :3]) < 0.5 for h in range(H)])
        r = dict(iters=it, extrapolate=None if ex is None else dict(angle_deg=ex[0], vmax_scale=ex[1]), tolerance=None if st is None else dict(tol_t=st[0], tol_r_deg=st[1], window=st[2]),
                 ms_per_step=float(np.median(ms)), ms_min=float(ms.min()), ms_max=float(ms.max()), ms_all=ms.tolist(),
                 hyp_per_s=H / (float(np.median(ms)) * 1e-3), best=best, best_rmse=float(rmse[best]),
                 winner_vs_gt=dict(centroid_mm=float(np.linalg.norm((c @ Tb[:3, :3] + Tb[3, :3]) - (c @ T_gt[:3, :3] + T_gt[3, :3]))),
                                   rot_fro=float(np.linalg.norm(Tb[:3, :3] - T_gt[:3, :3]))),
                 success_share=float(ok.mean()),
                 n_extrap_mean=float(b.n_extrap.cpu().numpy().mean()) if ex is not None else 0.0)
        if st is not None:
            r["n_iter_mean"] = float(b.n_iter.cpu().numpy().mean())
        res[s] = r
    m.destroy()
    return dict(workload=w["desc"], hypotheses=H, source_points=ns, model_points=w["nm"], settings=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--c4-hyp", type=int, default=bench.C4["hyp"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_icp_extrap.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("icp_extrap_bench.py: no CUDA device (there is no CPU path)")
    import pcreg_b200 as P
    P.init(0)
    out = dict(card=card(), steps=args.steps, warmup=args.warmup,
               l2="flushed: %d MB written before every timed step, outside its CUDA-event bracket" % (bench.L2_FLUSH_BYTES >> 20),
               schedule="settings alternated within each round; median of the steps", workloads={})
    out["workloads"]["c3"] = run_workload(P, torch, *c3_inputs(), args.steps, args.warmup)
    print(json.dumps(out["workloads"]["c3"]["settings"]), flush=True)
    out["workloads"]["c4_polish"] = run_workload(P, torch, *c4_inputs(args.c4_hyp), args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
