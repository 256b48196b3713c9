"""One windowed ICP call (include/pcreg.h: pcreg_icp_batch_windows_dev) against a loop of one call per window, on the reference
drivers' shape: 21 matching windows (slideMatchingWindow_v2.m:178-198) polished against C3's 10^6-point model.

    python tools/icp_windows_bench.py [--steps 3] [--warmup 1] [--out profiles/r07_icp_windows.json]

Windows: synth.make_source sources of 2 000 - 6 000 points (sigma 0.3), KNN mode (85 % trim), 30 iterations, grid NN on the voxel
map.  H_w in {1, 16, 256} hypotheses per window (synth.pose_grid around each window's truth).  Settings, alternated within each
round, every step through a device entry with bench.py's 256 MB L2 flush before it, outside the CUDA-event bracket:
  windows        one pcreg_icp_batch_windows_dev call, path chosen by the library's rule
  windows_fused  the same call with PCREG_FUSED=1 (one fused launch)       (H_w = 1 and 16)
  windows_loop   the same call with PCREG_FUSED=0 (loop over the windows)  (H_w = 1 and 16)
  loop21         21 pcreg_icp_batch_dev calls, one per window (each picks its own path as it always has)
The outputs (T, rmse, n_used, status, best per window) of every setting are compared bit for bit with loop21's.  The card name and
power limit are read in the same run.  Needs a GPU; there is no CPU path.
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

import bench  # noqa: E402  (C3 workload, L2 flush, timing brackets)
from icp_stop_bench import card  # noqa: E402

NWIN = 21
GRIDS = {1: (2, (1, 1, 1)), 16: (4, (2, 2, 1)), 256: (16, (4, 2, 2))}     # (rotations, translation lattice); H_w = 1 drops the unrotated pose


def make_windows(model, seed=2024):
    from pcreg_b200 import synth
    g = synth.rng(seed)
    wins = []
    for w in range(NWIN):
        src, T_gt, c = synth.make_source(model, int(g.integers(2000, 6001)), 0.3, seed + 1 + w)
        wins.append((src, T_gt, c))
    return wins


def run_batch(P, torch, m, wins, H, steps, warmup):
    from pcreg_b200 import synth, torch_ops
    dev = torch.device("cuda", 0)
    n_rot, tr = GRIDS[H]
    T0s = [synth.pose_grid(T_gt, c, n_rot, tr, 10.0, 1.0, 3000 + k)[-H:] for k, (_, T_gt, c) in enumerate(wins)]
    ns = np.array([s.shape[0] for s, _, _ in wins], dtype=np.int64)
    soff = np.concatenate([[0], np.cumsum(ns)]).astype(np.int64)
    hoff = np.arange(NWIN + 1, dtype=np.int64) * H
    iters = bench.WORKLOADS["c3"]["iters"]
    opts = P.icp_opts(mode=P.ICP_KNN, iters=iters, k_frac=0.85, nn=P.NN_GRID)
    src_cm = torch_ops.src_to_abi_t(torch.from_numpy(np.concatenate([s for s, _, _ in wins])).to(dev))
    T0_abi = torch_ops.T_to_abi_t(torch.from_numpy(np.concatenate(T0s)).to(dev)).reshape(-1, 16).contiguous()
    per_src = [torch_ops.src_to_abi_t(torch.from_numpy(s).to(dev)) for s, _, _ in wins]
    per_T0 = [T0_abi[k * H:(k + 1) * H] for k in range(NWIN)]
    settings = ["windows", "loop21"] + (["windows_fused", "windows_loop"] if H <= 16 else [])
    env = dict(windows=None, windows_fused="1", windows_loop="0", loop21=None)
    bufs = {s: torch_ops.IcpWindowsDeviceBuffers(NWIN * H, 0, NWIN, iters, dev) for s in settings if s != "loop21"}
    lbufs = [torch_ops.IcpDeviceBuffers(H, int(ns[k]), iters, dev) for k in range(NWIN)]
    flush = bench.Flusher(torch, dev)
    path = {}

    def step(s):
        if s == "loop21":
            for k in range(NWIN):
                torch_ops.icp_batch_device(m, per_src[k], None, per_T0[k], opts, lbufs[k])
            return
        if env[s] is None:
            os.environ.pop("PCREG_FUSED", None)
        else:
            os.environ["PCREG_FUSED"] = env[s]
        try:
            torch_ops.icp_windows_device(m, src_cm, soff, None, T0_abi, hoff, opts, bufs[s])
        finally:
            os.environ.pop("PCREG_FUSED", None)

    for s in settings:                                            # which path each windowed setting took
        if s != "loop21":
            P.set_profiling(2)
            step(s)
            path[s] = "fused" if P.last_profile()["fused"] == 1.0 else "loop"
            P.set_profiling(False)
    for _ in range(warmup):
        for s in settings:
            step(s)
    torch.cuda.synchronize()
    times = {s: [] for s in settings}
    for _ in range(steps):
        for s in settings:
            times[s] += bench.time_steps(torch, lambda: step(s), 1, flush, torch.cuda.synchronize)
    ref = dict(T=torch.cat([b.T for b in lbufs]).cpu().numpy(), rmse=torch.cat([b.rmse for b in lbufs]).cpu().numpy(),
               n_used=torch.cat([b.n_used for b in lbufs]).cpu().numpy(), status=torch.cat([b.status for b in lbufs]).cpu().numpy(),
               best=torch.cat([b.best for b in lbufs]).cpu().numpy())
    res = {}
    for s in settings:
        ms = np.asarray(times[s])
        r = dict(ms_per_step=float(np.median(ms)), ms_min=float(ms.min()), ms_max=float(ms.max()), ms_all=ms.tolist())
        if s != "loop21":
            b = bufs[s]
            got = dict(T=b.T.cpu().numpy(), rmse=b.rmse.cpu().numpy(), n_used=b.n_used.cpu().numpy(), status=b.status.cpu().numpy(),
                       best=b.best.cpu().numpy())
            r["bit_equal_to_loop21"] = all(np.array_equal(got[k], ref[k], equal_nan=got[k].dtype.kind == "f") for k in ref)
            r["path"] = path[s]
        res[s] = r
    for s in res:
        res[s]["speedup_vs_loop21"] = res["loop21"]["ms_per_step"] / res[s]["ms_per_step"]
    return dict(hyp_per_window=H, hypotheses=NWIN * H, source_points=ns.tolist(), settings=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_icp_windows.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("icp_windows_bench.py: no CUDA device (there is no CPU path)")
    import pcreg_b200 as P
    from pcreg_b200 import synth
    P.init(0)
    c3 = bench.WORKLOADS["c3"]
    model = synth.make_model(c3["nm"], c3["seed"])
    m = P.Model(model, grid=True)
    wins = make_windows(model)
    out = dict(card=card(), steps=args.steps, warmup=args.warmup, windows=NWIN, model_points=c3["nm"], mode="knn", iters=c3["iters"],
               l2="flushed: %d MB written before every timed step, outside its CUDA-event bracket" % (bench.L2_FLUSH_BYTES >> 20),
               schedule="settings alternated within each round", batches={})
    for H in sorted(GRIDS):
        out["batches"][str(H)] = run_batch(P, torch, m, wins, H, args.steps, args.warmup)
        print(json.dumps({H: {s: (r["ms_per_step"], r.get("path"), r.get("bit_equal_to_loop21")) for s, r in out["batches"][str(H)]["settings"].items()}}),
              flush=True)
    m.destroy()
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
