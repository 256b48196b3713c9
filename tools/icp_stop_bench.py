"""What the ICP convergence tolerance (include/pcreg.h: pcreg_icp_stop) buys on the C3 and C4 workloads of bench.py.

    python tools/icp_stop_bench.py [--steps 3] [--c4-hyp 100000] [--out profiles/r03_icp_stop.json]

For each workload the settings (no stop, the default {0.01, 0.5, 3}, a tighter {0.001, 0.05, 3}) are timed ALTERNATELY in one
process (round r times every setting once), each step through the device entry (pcreg_icp_batch{,_stop}_dev) with bench.py's
256 MB L2 flush before it, outside the CUDA-event bracket.  Reported per setting: ms per step (median, min, max), hypotheses/s,
the n_iter distribution, the converged fraction, the best rmse, and how far the winner's pose is from the no-stop winner's.
The card name and power limit are read in the same run.  Needs a GPU; there is no CPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload definitions, L2 flush, timing brackets)

SETTINGS = [("none", None), ("default", (0.01, 0.5, 3)), ("tight", (0.001, 0.05, 3))]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clk)


def c3_inputs():
    w = bench.WORKLOADS["c3"]
    model, src, T0, w_src, _ = bench.make_inputs(w, 0)
    return w, model, src, T0, w_src, dict(mode="knn", thDist2=0.0)


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
    return w, model, src, T0, None, dict(mode="plain", thDist2=c["thDist2"])


def run_workload(P, torch, name, w, model, src, T0, w_src, mkw, steps, warmup):
    from pcreg_b200 import torch_ops
    dev = torch.device("cuda", 0)
    m = P.Model(model, grid=True)
    mode = dict(plain=P.ICP_PLAIN, knn=P.ICP_KNN, weighted=P.ICP_WEIGHTED)[mkw["mode"]]
    opts = P.icp_opts(mode=mode, iters=w["iters"], k_frac=0.85, R_w=3.5, thDist2=mkw["thDist2"], nn=P.NN_GRID)
    H, ns = T0.shape[0], src.shape[0]
    src_cm = torch_ops.src_to_abi_t(torch.from_numpy(src).to(dev))
    T0_abi = torch_ops.T_to_abi_t(torch.from_numpy(T0).to(dev))
    w_t = torch.from_numpy(w_src).to(dev) if w_src is not None else None
    flush = bench.Flusher(torch, dev)
    bufs = {s: torch_ops.IcpDeviceBuffers(H, ns, w["iters"], dev, want_n_iter=st is not None) for s, st in SETTINGS}
    stops = {s: (P.icp_stop(*st) if st is not None else None) for s, st in SETTINGS}

    def step(s):
        torch_ops.icp_batch_device(m, src_cm, w_t, T0_abi, opts, bufs[s], stop=stops[s])

    for _ in range(warmup):
        for s, _ in SETTINGS:
            step(s)
    torch.cuda.synchronize()
    times = {s: [] for s, _ in SETTINGS}
    for _ in range(steps):                                        # alternate: one step of every setting per round
        for s, _ in SETTINGS:
            times[s] += bench.time_steps(torch, lambda: step(s), 1, flush, torch.cuda.synchronize)
    res = {}
    ref_T = None
    for s, st in SETTINGS:
        b = bufs[s]
        T = torch_ops.T_from_abi_t(b.T).cpu().numpy()
        rmse = b.rmse.cpu().numpy()
        best = int(b.best.item())
        ms = np.asarray(times[s])
        r = dict(tolerance=None if st is None else dict(tol_t=st[0], tol_r_deg=st[1], window=st[2]),
                 ms_per_step=float(np.median(ms)), ms_min=float(ms.min()), ms_max=float(ms.max()), ms_all=ms.tolist(),
                 hyp_per_s=H / (float(np.median(ms)) * 1e-3), best=best, best_rmse=float(rmse[best]))
        if st is None:
            ref_T = T[best]
            r.update(n_iter=dict(mean=float(w["iters"]), p50=w["iters"], p90=w["iters"], max=w["iters"]), converged_frac=0.0)
        else:
            n = b.n_iter.cpu().numpy()
            r.update(n_iter=dict(mean=float(n.mean()), p50=float(np.percentile(n, 50)), p90=float(np.percentile(n, 90)), max=int(n.max())),
                     converged_frac=float(b.converged.cpu().numpy().mean()))
        r["winner_vs_no_stop"] = dict(rot_fro=float(np.linalg.norm(T[best][:3, :3] - ref_T[:3, :3])),
                                      trans=float(np.linalg.norm(T[best][3, :3] - ref_T[3, :3])))
        res[s] = r
    base = res["none"]["ms_per_step"]
    for s in res:
        res[s]["speedup_vs_no_stop"] = base / res[s]["ms_per_step"]
    m.destroy()
    return dict(workload=w["desc"], hypotheses=H, source_points=ns, model_points=w["nm"], iters=w["iters"], settings=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--c4-hyp", type=int, default=bench.C4["hyp"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_icp_stop.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("icp_stop_bench.py: no CUDA device (there is no CPU path)")
    import pcreg_b200 as P
    P.init(0)
    out = dict(card=card(), steps=args.steps, warmup=args.warmup,
               l2="flushed: %d MB written before every timed step, outside its CUDA-event bracket" % (bench.L2_FLUSH_BYTES >> 20),
               schedule="settings alternated within each round", workloads={})
    out["workloads"]["c3"] = run_workload(P, torch, "c3", *c3_inputs(), args.steps, args.warmup)
    print(json.dumps(out["workloads"]["c3"]["settings"]), flush=True)
    out["workloads"]["c4_polish"] = run_workload(P, torch, "c4", *c4_inputs(args.c4_hyp), args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
