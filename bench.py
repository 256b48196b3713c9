#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric (ICP NN queries/s & aligned hypotheses/s) on N B200s.

One "step" = one full multi-start ICP job over the workload's hypothesis batch.  Headline workload = BASELINE.json
configs[2] (C3): 4096 initial poses PER GPU (weak scaling: one global pose grid dealt round-robin to the ranks, no
data-path collective; the final all-gather of result records and the arg-min are inside the timed region), 5k-point
source vs 1M-point model, KNN-trimmed ICP, 30 iterations, grid NN (Voronoi voxel map + fused per-hypothesis kernel).

  value   device-resident inputs through pcreg_icp_batch_dev, CUDA events around every step, max over ranks
  e2e     the same job through the host-buffer C-ABI call pcreg_icp_batch (pinned host inputs, H2D + D2H inside the timed
          region); at N > 1 it is ONE process (rank 0) driving all N GPUs through pcreg_init(devices, N) -- the library shards
          the hypotheses itself (include/pcreg.h) -- while the other ranks wait on a host-side barrier
  strong  BASELINE.json's literal config 3 (4096 poses in TOTAL, 4096 / N per GPU) beside the weak-scaling headline

At N = 1 the other configurations are measured beside the headline (bounded, each skippable with --no-<name>):
  c2 (configs[1]: one weighted alignment, brute-force NN, FP32-FMA roofline; + the same through the grid path),
  c4 (configs[3]: 10^5 RANSAC hypotheses scored + 10^5 seeded poses polished by 20 ICP iterations, 20k vs 2M),
  c5 (configs[4]: one GPU's share -- 2048 poses x 65 536 source points vs a 16M-point model, not L2-resident),
  get_matches (row f4), align_batch (rows a1-a5: AlignPoints family over thousands of neighbourhoods), cpu_baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c3|c2|c2g|c5|small] [--dump-outputs DIR]

--impl reference times the CPU oracle restatement (the reference is MATLAB; MATLAB/Octave are probed and reported, neither
exists in this image) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FFMA_PEAK_TFLOPS_MEASURED = 65.7      # tools/fma_peak.cu on this pool's B200 (profiles/r01_fma_peak.txt)
HBM_FALLBACK_GBS = 6650.0             # /opt/skills/guides/B200_PROFILING.md fallback
L2_FLUSH_BYTES = 256 << 20            # written between timed steps (L2 is 126 MB)

WORKLOADS = {
    # name: nm, ns, hyps per GPU, iters, mode, nn, pose grid (n_rot, (nx,ny,nz)), max_deg, sigma, seed
    "c3": dict(nm=1_000_000, ns=5000, hyp=4096, iters=30, mode="knn", nn="grid", rot=16, trans=(8, 8, 4), max_deg=20.0,
               sigma=0.3, seed=1003, desc="C3 multi-start ICP: 4096 poses/GPU x 5k src vs 1M model, KNN-trimmed, 30 it, grid NN"),
    "c2": dict(nm=500_000, ns=10_000, hyp=1, iters=100, mode="weighted", nn="brute", rot=1, trans=(1, 1, 1), max_deg=0.0,
               sigma=0.3, seed=1002, desc="C2 AlignPoints_weighted-style single alignment: 10k weighted src vs 500k model, 100 it, brute NN"),
    "c2g": dict(nm=500_000, ns=10_000, hyp=1, iters=100, mode="weighted", nn="grid", rot=1, trans=(1, 1, 1), max_deg=0.0,
                sigma=0.3, seed=1002, desc="C2 with the grid NN path (same inputs and results as C2, what a user would run)"),
    # one GPU's share of BASELINE.json configs[4] (16k hypotheses over 8 GPUs): the model (512 MB of points + grid) is NOT
    # L2-resident; band-limited voxel map (15.5 GB) + per-pass kernels (65 536 source points do not fit the fused kernel)
    "c5": dict(nm=16_000_000, ns=65536, hyp=2048, iters=20, mode="knn", nn="grid", rot=8, trans=(8, 8, 4), max_deg=10.0,
               sigma=0.3, seed=1005, src_stride=16,
               desc="C5 large upsampled model: 2048 poses/GPU x 65 536 src vs 16M model, KNN-trimmed, 20 it, grid NN"),
    "small": dict(nm=100_000, ns=2000, hyp=256, iters=10, mode="knn", nn="grid", rot=4, trans=(4, 4, 4), max_deg=10.0,
                  sigma=0.3, seed=7, desc="small multi-start ICP (debug)"),
}
C4 = dict(nm=2_000_000, ns=20_000, hyp=100_000, iters=20, P=600, inlier_frac=0.25, sigma_match=0.15, thDist=0.3, ratio=0.08,
          thDist2=4.0, seed=1004,
          desc="C4 RANSAC-seeded refinement: 10^5 hypotheses scored on 600 putative matches (refit on inliers), 10^5 seeded poses "
               "polished by 20 ICP iterations (PLAIN, thDist2 = 4), 20k src vs 2M model, grid NN")


def make_inputs(w, rank, world=1):
    """Synthetic inputs of workload w for one rank.  Multi-GPU (weak scaling): ONE pose grid of hyp * world poses --
    the same rotations, the z lattice refined `world` times over the same extent -- dealt to the ranks round-robin,
    so that every GPU gets a statistically identical share."""
    from pcreg_b200 import synth
    model = synth.make_model(w["nm"], w["seed"])
    src, T_gt, c = synth.make_source(model[::w.get("src_stride", 1)], w["ns"], w["sigma"], w["seed"])
    if w["hyp"] == 1:
        T0 = synth.perturb_pose(T_gt, c, synth.rot_axis_angle([0.3, -0.5, 0.8], np.deg2rad(5.0)), np.array([1.2, -1.0, 1.2]))[None]
    else:
        nx, ny, nz = w["trans"]
        T0 = synth.pose_grid(T_gt, c, w["rot"], (nx, ny, nz * world), w["max_deg"], (2.0, 2.0, 2.0 / world), w["seed"])
        T0 = np.ascontiguousarray(T0[rank::world][: w["hyp"]])
    g = synth.rng(w["seed"] + 5)
    w_src = g.uniform(0.5, 1.0, w["ns"]) if w["mode"] == "weighted" else None
    return model, src, T0, w_src, T_gt


def config_of(w, hyp=None, world=1):
    """The workload-defining part of the JSON line: identical in the GPU arm and in the reference arm."""
    return dict(workload=w["desc"], hypotheses_per_gpu=int(hyp if hyp is not None else w["hyp"]), source_points=w["ns"],
                model_points=w["nm"], iters=w["iters"], mode=w["mode"], nn=w["nn"],
                parallelism="hypotheses sharded over the GPUs, model replicated, final gather of result records + first-index arg-min",
                l2="flushed: %d MB written between timed steps, outside the per-step CUDA-event brackets (L2 is 126 MB)" % (L2_FLUSH_BYTES >> 20))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        exe = shutil.which("nvidia-smi")
        if not exe:
            return
        self.proc = subprocess.Popen([exe, "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples in the timed region"], samples=0)
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json, STREAM-style copy)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


# the sources of the kernels whose DRAM traffic profiles/roofline_traffic.json records
TRAFFIC_SOURCES = ("icp.cu", "icp_fused.cu", "nn_brute.cu", "nn_grid.cu", "nn_vox.cu", "pcreg_dev.cuh", "pcreg_grid.cuh", "pcreg_icp.cuh",
                   "pcreg_math.cuh", "pcreg_select.cuh", "pcreg_vox.cuh")


def kernel_source_sha():
    """Hash of the CUDA sources: profiles/roofline_traffic.json is only used while it matches the code it was captured from."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "pcreg_b200", "csrc")
    for name in TRAFFIC_SOURCES:
        with open(os.path.join(d, name), "rb") as f:
            h.update(name.encode()); h.update(f.read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel from the committed ncu --set full
    capture -- or None when the capture was taken from other sources than the ones being run (stale)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        with open(p) as f:
            d = json.load(f)
        if d.get("csrc_sha16") != kernel_source_sha():
            return None
        return d.get("kernels", {}).get(kernel)
    except Exception:
        return None


def probe_matlab():
    return [x for x in ("matlab", "octave", "octave-cli") if shutil.which(x)]


# ----------------------------------------------------------------------------------------------
# CPU arm (oracle restatement): bounded sample of the same workload
# ----------------------------------------------------------------------------------------------
def cpu_sample(w, budget_s=12.0, max_hyp=None):
    import oracle
    model, src, T0, w_src, _ = make_inputs(w, 0)
    omode = dict(plain=oracle.ICP_PLAIN, knn=oracle.ICP_KNN, weighted=oracle.ICP_WEIGHTED)[w["mode"]]
    t_build0 = time.perf_counter()
    nn = oracle.nn.KDTreeNN(np.asarray(model, dtype=np.float64))
    t_build = time.perf_counter() - t_build0
    n = 0
    t0 = time.perf_counter()
    limit = T0.shape[0] if max_hyp is None else min(max_hyp, T0.shape[0])
    while n < limit:
        oracle.icp_single(model, src, T0[n], mode=omode, iters=w["iters"], k_frac=0.85, R_w=3.5, w_src=w_src, nn=nn)
        n += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    q = n * w["ns"] * (w["iters"] + 1)
    return dict(queries_per_s=q / dt, hyp_per_s=n / dt, n_hyp=n, seconds=dt, kdtree_build_s=t_build)


def run_reference(args, w, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    vals = []
    for _ in range(args.warmup):
        cpu_sample(w, budget_s=1.0, max_hyp=1)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        vals.append(cpu_sample(w, budget_s=max(2.0, 60.0 / max(1, args.steps))))
    dt = time.perf_counter() - t0
    v = float(np.mean([x["queries_per_s"] for x in vals]))
    sample = "%d hypotheses/step of the %s workload (oracle restatement: numpy FP64 + scipy cKDTree workers=-1; %s)" % (
        vals[-1]["n_hyp"], args.workload,
        "MATLAB/Octave not installed" if not probe_matlab() else "found " + ",".join(probe_matlab()) + " but the composed ICP has no .m file")
    line = dict(impl="reference", metric="ICP NN queries/s", value=v, unit="queries/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * dt / max(1, args.steps), higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic", config=config_of(w, world=world),
                hyp_per_s=float(np.mean([x["hyp_per_s"] for x in vals])),
                cpu_baseline=dict(value=v, unit="queries/s", cores=cores, kind="port", sample=sample),
                e2e=dict(value=v, unit="queries/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
class Flusher:
    def __init__(self, torch, dev):
        self.buf = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def __call__(self):
        self.buf.fill_(1)


def time_steps(torch, fn, steps, flush, sync_all):
    """fn() `steps` times, an L2 flush before each, one CUDA-event bracket per step.  Returns the list of ms."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    sync_all()
    for a, b in ev:
        flush()
        a.record()
        fn()
        b.record()
    sync_all()
    return [a.elapsed_time(b) for a, b in ev]


def gpu_workload(P, torch, w, rank, steps, warmup, dist=None, world=1, T0_override=None, do_e2e=True, do_profile=True, opts_kw=None,
                 inputs=None, keep_outputs=False):
    """Measurements of one workload on this rank (collectives included when world > 1).  keep_outputs: r["outputs"] holds
    what the last timed step returned, copied to the host before any untimed step reuses the buffers."""
    from pcreg_b200 import sharded, torch_ops
    dev = torch.device("cuda", torch.cuda.current_device())
    # PCREG_BENCH_SHARD="r/n": measure on ONE GPU the share that rank r of an n-GPU run would get (work-balance check)
    shard = os.environ.get("PCREG_BENCH_SHARD")
    in_rank, in_world = (int(shard.split("/")[0]), int(shard.split("/")[1])) if shard else (rank, world)
    model_h, src, T0, w_src, T_gt = inputs if inputs is not None else make_inputs(w, in_rank, in_world)
    if T0_override is not None:
        T0 = T0_override
    m = P.Model(model_h, grid=(w["nn"] == "grid"), cells_per_point=float(os.environ.get("PCREG_GRID_CPP", "0")))
    mode = dict(plain=P.ICP_PLAIN, knn=P.ICP_KNN, weighted=P.ICP_WEIGHTED)[w["mode"]]
    nn = P.NN_GRID if w["nn"] == "grid" else P.NN_BRUTE
    opts = P.icp_opts(mode=mode, iters=w["iters"], k_frac=0.85, R_w=3.5, nn=nn, **(opts_kw or {}))
    H, ns = T0.shape[0], src.shape[0]
    src_cm = torch_ops.src_to_abi_t(torch.from_numpy(src).to(dev))
    T0_abi = torch_ops.T_to_abi_t(torch.from_numpy(T0).to(dev))
    w_t = torch.from_numpy(w_src).to(dev) if w_src is not None else None
    out = torch_ops.IcpDeviceBuffers(H, ns, w["iters"], dev)
    flush = Flusher(torch, dev)
    h_best = torch.empty(1, dtype=torch.int64).pin_memory()

    def step_device():
        torch_ops.icp_batch_device(m, src_cm, w_t, T0_abi, opts, out)
        if world > 1:
            rec = torch.cat([out.rmse[:, None], out.T, out.n_used[:, None].double(), out.status[:, None].double()], dim=1)
            _, best = sharded.gather_and_pick(rec, H * world, H, on_device=True)
            h_best.copy_(best.reshape(1), non_blocking=True)           # the step's result read: winner index, 8 bytes
        else:
            h_best.copy_(out.best, non_blocking=True)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(warmup):
        step_device()
    sync_all()
    launches0 = P.launch_count()
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    time.sleep(0.25)
    t_wall0 = time.time()
    per_step = time_steps(torch, step_device, steps, flush, sync_all)
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1)
    launches = P.launch_count() - launches0
    outputs = None
    if keep_outputs:
        # T: [H, 16] column-major 4x4 records as pcreg_icp_batch_dev writes them; best: the step's winner index
        outputs = {k: v.cpu().numpy().astype(np.float64)
                   for k, v in dict(T=out.T, rmse=out.rmse, n_used=out.n_used, status=out.status, best=h_best).items()}
    ms = float(sum(per_step))
    ms_ranks = [ms / steps]
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        allms = torch.empty(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allms, tt)
        ms_ranks = [float(x) / steps for x in allms.cpu()]
        ms = max(ms_ranks) * steps
    rmse_best = float(out.rmse[int(out.best.item())].item())
    r = dict(ms_per_step=ms / steps, q_per_step=H * ns * (w["iters"] + 1), H=H, ns=ns, launches=launches, clocks=clocks,
             ms_ranks=ms_ranks, rmse_best=rmse_best, nm=model_h.shape[0], per_step_ms=per_step, outputs=outputs)
    if do_profile:
        # two extra UNTIMED steps: (2) CUDA-event times of the kernels with nothing added to them, (1) exact device-side work
        # counters (atomics inside the kernels) and the phase clocks of the fused kernel
        P.set_profiling(2)
        step_device(); sync_all()
        r["prof_t"] = P.last_profile()
        P.set_profiling(1)
        step_device(); sync_all()
        r["prof"] = P.last_profile()
        P.set_profiling(False)
    if do_e2e:
        r.update(e2e_single_device(P, torch, m, src, T0, w_src, opts, flush, out, steps))
    r["grid"] = None
    if w["nn"] == "grid":
        r["grid"] = m.grid_info()
        r["grid"]["voxel_map"] = m.voxel_info()
    m.destroy()
    return r


def pinned_inputs(torch, src, T0, w_src):
    H = T0.shape[0]
    h = dict(src=torch.from_numpy(np.asfortranarray(src).T.copy()).pin_memory(),            # [3, ns] = column-major ns x 3
             T0=torch.from_numpy(np.ascontiguousarray(np.swapaxes(T0, 1, 2))).pin_memory(),
             w=torch.from_numpy(w_src).pin_memory() if w_src is not None else None,
             T=torch.empty((H, 16), dtype=torch.float64).pin_memory(), rmse=torch.empty(H, dtype=torch.float64).pin_memory(),
             nu=torch.empty(H, dtype=torch.int32).pin_memory(), st=torch.empty(H, dtype=torch.int32).pin_memory())
    h["h2d"] = h["src"].numel() * 8 + h["T0"].numel() * 8 + (h["w"].numel() * 8 if h["w"] is not None else 0)
    h["d2h"] = h["T"].numel() * 8 + h["rmse"].numel() * 8 + h["nu"].numel() * 4 + h["st"].numel() * 4 + 8
    return h


def host_call(P, m, h, ns, H, opts):
    import ctypes as C
    from pcreg_b200 import _lib as L
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    cast = lambda t, ty: C.cast(C.c_void_p(t.data_ptr()), ty) if t is not None else None
    best = C.c_int64()
    L.check(L.lib().pcreg_icp_batch(m.handle, vp(h["src"]), 1, ns, ns, cast(h["w"], L.c_f64p), cast(h["T0"], L.c_f64p), H, C.byref(opts),
                                    cast(h["T"], L.c_f64p), cast(h["rmse"], L.c_f64p), cast(h["nu"], L.c_i32p), cast(h["st"], L.c_i32p),
                                    None, None, C.byref(best)), "pcreg_icp_batch")
    return int(best.value)


def e2e_single_device(P, torch, m, src, T0, w_src, opts, flush, out, steps):
    """The public host-buffer API on this rank's GPU: pinned host inputs, H2D + D2H inside the timed region."""
    H, ns = T0.shape[0], src.shape[0]
    h = pinned_inputs(torch, src, T0, w_src)
    host_call(P, m, h, ns, H, opts)
    ms = time_steps(torch, lambda: host_call(P, m, h, ns, H, opts), steps, flush, torch.cuda.synchronize)
    ok = bool(np.array_equal(h["rmse"].numpy(), out.rmse.cpu().numpy(), equal_nan=True))
    return dict(ms_per_step_e2e=float(np.mean(ms)), h2d=h["h2d"], d2h=h["d2h"], e2e_equals_device=ok)


def e2e_multi_device(P, torch, w, world, steps):
    """N > 1, rank 0 only: ONE process drives all N GPUs through the C ABI (pcreg_init(devices, N); pcreg_icp_batch shards the
    N * 4096 hypotheses over the devices inside the library).  Host wall clock around the synchronous call, every device
    synchronised and its L2 flushed before each step."""
    from pcreg_b200 import synth
    model_h, src, _, w_src, T_gt = make_inputs(w, 0, 1)
    _, _, c = synth.make_source(model_h[::w.get("src_stride", 1)], w["ns"], w["sigma"], w["seed"])
    nx, ny, nz = w["trans"]
    grid = synth.pose_grid(T_gt, c, w["rot"], (nx, ny, nz * world), w["max_deg"], (2.0, 2.0, 2.0 / world), w["seed"])
    T0 = np.ascontiguousarray(np.concatenate([grid[r::world][: w["hyp"]] for r in range(world)]))      # the ranks' shares, rank-major
    P.init(list(range(world)))
    m = P.Model(model_h, grid=(w["nn"] == "grid"))
    mode = dict(plain=P.ICP_PLAIN, knn=P.ICP_KNN, weighted=P.ICP_WEIGHTED)[w["mode"]]
    opts = P.icp_opts(mode=mode, iters=w["iters"], k_frac=0.85, R_w=3.5, nn=P.NN_GRID if w["nn"] == "grid" else P.NN_BRUTE)
    H, ns = T0.shape[0], src.shape[0]
    h = pinned_inputs(torch, src, T0, w_src)
    flushers = []
    for d in range(world):
        with torch.cuda.device(d):
            flushers.append(Flusher(torch, torch.device("cuda", d)))

    def sync_flush():
        for d, f in enumerate(flushers):
            with torch.cuda.device(d):
                f()
        for d in range(world):
            torch.cuda.synchronize(d)

    host_call(P, m, h, ns, H, opts)
    host_call(P, m, h, ns, H, opts)
    ts = []
    for _ in range(steps):
        sync_flush()
        t0 = time.perf_counter()
        best = host_call(P, m, h, ns, H, opts)
        ts.append(1e3 * (time.perf_counter() - t0))
    rmse_best = float(h["rmse"][best])
    m.destroy()
    P.init(int(os.environ.get("LOCAL_RANK", "0")))
    return dict(ms_per_step_e2e=float(np.mean(ts)), h2d=h["h2d"], d2h=h["d2h"], rmse_best=rmse_best, H=H,
                how="one process, pcreg_init(devices 0..%d), pcreg_icp_batch with pinned host buffers; host wall clock "
                    "around the synchronous call (it returns after every device has copied its records back)" % (world - 1))


def roofline_for(w, r):
    """Roofline of the dominant kernel of the workload: algorithmic bytes (DESIGN.md section 3) from the exact device-side
    work counters of one profiled step, divided by the kernel's CUDA-event time of another profiled step that ran WITHOUT the
    counters (their atomics slow the kernels down)."""
    p, pt = r["prof"], r["prof_t"]
    peak, how = hbm_peak()
    if w["nn"] == "grid" and p.get("fused"):
        # k_icp_fused, all passes of all hypotheses in one launch.  Per query and pass: NN = 24 B source point + 8 B voxel header
        # + 16 B per list entry scanned + 32 B per point gathered for the FP64 decision; sums = 24 B source point + 32 B model
        # point (+ 8 B weight) per SELECTED correspondence.  Correspondences and trim keys never leave shared memory.
        nq = p["nn_queries"]
        sel = 0.85 if w["mode"] == "knn" else 1.0       # trimmed mode: the sums pass reads only the selected correspondences (k_frac)
        by = nq * (24.0 + 8.0) + nq * sel * (24.0 + 32.0 + (8.0 if w["mode"] == "weighted" else 0.0)) + 16.0 * p["list_entries_read"] \
            + 32.0 * p["list_points_gathered"] + 36.0 * p["walked_queries"]
        ms = pt["nn_ms"]
        gbs = by / max(ms, 1e-9) / 1e6
        return dict(bound="hbm", kernel="k_icp_fused", achieved=gbs, peak=peak, unit="GB/s", frac=gbs / peak, traffic=ncu_traffic("k_icp_fused"),
                    peak_source=how, bytes_per_launch=by, avg_launch_ms=ms, launches_per_step=1,
                    note="one launch per step; algorithmic bytes from exact device-side counters; the lists a converging batch touches "
                         "stay L2-resident, so DRAM traffic (traffic, from ncu) is below the algorithmic bytes and the kernel is bound by "
                         "L1 wavefronts of its scattered 16-byte loads and by the block-wide phases of a hypothesis, not by HBM",
                    phase_share=p["fused_phase_share"], entries_per_query=p["list_entries_read"] / max(1.0, nq),
                    fp64_points_per_query=p["list_points_gathered"] / max(1.0, nq), walked_fraction=p["walked_queries"] / max(1.0, nq))
    if w["nn"] == "grid" and p.get("voxel_map"):
        kern = {
            "k_nn_vox": dict(ms=pt["list_ms"], launches=pt["list_launches"],
                             bytes=8.0 * p["nn_queries"] + 36.0 * p["certified_queries"] + 16.0 * p["list_entries_read"] + 32.0 * p["list_points_gathered"]),
            "k_nn_grid_walk": dict(ms=pt["walk_ms"], launches=pt["walk_launches"],
                                   bytes=36.0 * p["walked_queries"] + 8.0 * p["walk_leaves"] + 32.0 * p["walk_points"]
                                         + 1.0 * max(0.0, p["grid_nodes_popped"] - p["walk_leaves"])),
            "k_icp_update": dict(ms=pt["update_ms"], launches=pt["update_launches"], bytes=76.0 * p["correspondences"]),
        }
    elif w["nn"] == "grid":
        nq_pass = r["H"] * r["ns"]
        kern = {
            # every query of the pass reads its 8-byte list descriptor; a scanned query also its 16-byte header, its
            # 24-byte source point and writes 12 bytes; 4 bytes per list entry read, 32 bytes per model point gathered
            "k_nn_list": dict(ms=pt["list_ms"], launches=pt["list_launches"],
                              bytes=8.0 * nq_pass * p["list_launches"] + 52.0 * p["certified_queries"] + 4.0 * p["list_entries_read"]
                                    + 32.0 * p["list_points_gathered"]),
            # 24-byte source point + 12-byte result per query, 8 bytes (start, end) per visited cell row, 32 bytes per point
            "k_nn_grid_rows": dict(ms=pt["rowscan_ms"], launches=pt["rowscan_launches"],
                                   bytes=36.0 * p["rowscan_queries"] + 8.0 * p["rowscan_rows"] + 32.0 * p["rowscan_points"]),
            # same per query / leaf / point, plus 1 mask byte per expanded pyramid node
            "k_nn_grid_walk": dict(ms=pt["walk_ms"], launches=pt["walk_launches"],
                                   bytes=36.0 * p["walked_queries"] + 8.0 * p["walk_leaves"] + 32.0 * p["walk_points"]
                                         + 1.0 * max(0.0, p["grid_nodes_popped"] - p["walk_leaves"])),
            "k_icp_update": dict(ms=pt["update_ms"], launches=pt["update_launches"], bytes=76.0 * p["correspondences"]),
        }
    else:
        pairs, launches = p["brute_pairs"], max(1.0, p["nn_launches"])
        achieved = 6.0 * pairs / (pt["nn_ms"] * 1e-3) / 1e12
        return dict(bound="fp32_fma", kernel="k_nn_brute", achieved=achieved, peak=FFMA_PEAK_TFLOPS_MEASURED, unit="TFLOP/s",
                    frac=achieved / FFMA_PEAK_TFLOPS_MEASURED, traffic=ncu_traffic("k_nn_brute"),
                    peak_source="measured FFMA microbenchmark tools/fma_peak.cu (theoretical 74.4 TFLOP/s at 1965 MHz)",
                    flops_per_launch=6.0 * pairs / launches, avg_launch_ms=pt["nn_ms"] / launches,
                    note="6 FLOP per (query, model point) pair; includes the bound pass and the FP64 slow path in the time")
    for k, v in kern.items():
        v["gbs"] = v["bytes"] / max(v["ms"], 1e-9) / 1e6
        v["frac"] = v["gbs"] / peak
        v["traffic"] = ncu_traffic(k)
    top = max(kern, key=lambda k: kern[k]["ms"])
    t = kern[top]
    launches = max(1.0, t["launches"])
    return dict(bound="hbm", kernel=top, achieved=t["gbs"], peak=peak, unit="GB/s", frac=t["frac"], traffic=t["traffic"],
                peak_source=how, bytes_per_launch=t["bytes"] / launches, avg_launch_ms=t["ms"] / launches,
                note="algorithmic bytes from exact device-side counters (DESIGN.md section 3); kernel times from a profiled step "
                     "without the counters",
                kernels={k: dict(ms=v["ms"], launches=v["launches"], algorithmic_bytes=v["bytes"], gbs=v["gbs"], frac=v["frac"],
                                 traffic=v["traffic"]) for k, v in kern.items()},
                list_answered_fraction=p["certified_queries"] / max(1.0, p["nn_queries"]))


def step_bytes(w, r):
    """Whole-step algorithmic bytes / measured step time / HBM peak."""
    rf = r.get("roofline") or {}
    if "kernels" in rf:
        by = sum(v["algorithmic_bytes"] for v in rf["kernels"].values())
    elif rf.get("unit") == "GB/s":
        by = rf["bytes_per_launch"] * rf.get("launches_per_step", 1)
    else:
        return None
    peak, _ = hbm_peak()
    gbs = by / (r["ms_per_step"] * 1e-3) / 1e9
    return dict(algorithmic_bytes_per_step=by, gbs=gbs, frac_of_hbm_peak=gbs / peak)


FP64_INST_PEAK_MEASURED = 16.45e12    # DFMA issue rate, tools/fma_peak.cu (32.9 TFLOP/s; profiles/r01_fma_peak.txt)


def match_workload(P, torch, n1=3000, n2=20000, dim=980, reps=3):
    """SURVEY.md section 8 row f4 beside the headline: getMatches (descriptor weighting + exhaustive matchFeatures) of n1 surface
    against n2 model descriptors through the host-buffer API.  The score kernel is FP64-pipe bound: 2 FP64 instructions
    per (pair, dimension) term for SAD."""
    g = np.random.default_rng(1)
    dS = g.poisson(g.gamma(0.6, 4.0, (n1, dim))).astype(np.float64)
    dM = g.poisson(g.gamma(0.6, 4.0, (n2, dim))).astype(np.float64)
    dM[::7][: n1 // 2] = dS[: n1 // 2]                                             # some exact partners, so matches exist
    par = dict(UNNORMALIZE=True, norm_factor=2, CHANGE_METRIC=True, metric_factor=0.6, MatchThreshold=10, MaxRatio=0.99,
               Metric="SAD", Unique=True)                                          # completeExperiment.m:112-122
    dS, dM = np.asfortranarray(dS), np.asfortranarray(dM)
    P.getMatches(dS[:64], dM[:64], par)
    launches0 = P.launch_count()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        matches = P.getMatches(dS, dM, par)
    wall_ms = (time.perf_counter() - t0) * 1e3 / reps
    launches = (P.launch_count() - launches0) // reps
    P.set_profiling(True)
    P.getMatches(dS, dM, par)
    pr = P.last_profile()
    P.set_profiling(False)
    inst_s = 2.0 * pr["match_terms"] / (pr["match_score_ms"] * 1e-3)
    return dict(workload="getMatches: %d surface x %d model descriptors, 981 dimensions, SAD, exhaustive matchFeatures" % (n1, n2),
                value=n1 * n2 / (wall_ms * 1e-3), unit="descriptor pairs/s (host buffers, H2D inside)", ms_per_call=wall_ms,
                h2d_bytes_per_call=int(dS.nbytes + dM.nbytes), matches=int(matches.shape[0]), gpu_launches=int(launches),
                roofline=dict(bound="fp64_pipe", kernel="k_match_scores", achieved=inst_s / 1e12, peak=FP64_INST_PEAK_MEASURED / 1e12,
                              unit="T FP64 inst/s", frac=inst_s / FP64_INST_PEAK_MEASURED, avg_launch_ms=pr["match_score_ms"],
                              terms_per_launch=pr["match_terms"],
                              note="2 FP64 instructions per (pair, dimension) term (t = a - b; acc += |t|); peak = measured DFMA issue rate"))


def align_batch_workload(P, torch, nb=10_000, reps=2):
    """Rows a1-a5 at the workload of visualizeGTMatches.m:94-141: thousands of neighbourhoods of 500-6000 points through the
    AlignPoints family, one batched call per variant (host buffers).  The kernel streams every neighbourhood: SURVEY.md
    section 8d byte model = 2 passes over the input + 1 output = 3 x 24 B per point (class double)."""
    from pcreg_b200 import synth
    base = synth.make_neighbourhoods((nb + 3) // 4, 77)                         # 4 shifted copies of each: generation is host time
    nbs = [a + np.array([17.0 * k, -9.0 * k, 4.0 * k]) for k in range(4) for a in base][:nb]
    npts = int(sum(a.shape[0] for a in nbs))
    peak, how = hbm_peak()
    out = {}
    for name, kind in (("AlignPoints", P.ALIGN_PLAIN), ("AlignPoints_KNN", P.ALIGN_KNN_FRAC), ("AlignPoints_weighted", P.ALIGN_WEIGHTED)):
        P.align_points_batch(kind, nbs[:8])
        t0 = time.perf_counter()
        for _ in range(reps):
            P.align_points_batch(kind, nbs)
        wall_ms = (time.perf_counter() - t0) * 1e3 / reps
        P.set_profiling(True)
        ks = []
        for _ in range(3):
            P.align_points_batch(kind, nbs)
            ks.append(P.last_profile()["match_score_ms"])                          # out[24]: ms of k_align_points
        P.set_profiling(False)
        kms = sorted(ks)[1]                                                        # median of three launches
        gbs = 72.0 * npts / max(kms, 1e-9) / 1e6
        out[name] = dict(neighbourhoods_per_s_host_call=nb / (wall_ms * 1e-3), ms_per_call=wall_ms, kernel_ms=kms,
                         roofline=dict(bound="hbm", kernel="k_align_points", achieved=gbs, peak=peak, unit="GB/s", frac=gbs / peak,
                                       bytes_per_launch=72.0 * npts, avg_launch_ms=kms, peak_source=how))
    return dict(workload="AlignPoints family, %d neighbourhoods of 500-6000 points (%d points, class double), one batched call per variant "
                         "(Python list marshaling included in ms_per_call)" % (nb, npts), variants=out)


def c4_workload(P, torch, steps=2):
    """BASELINE.json configs[3]: 10^5 getInliersRANSAC-style hypotheses scored (3-point Kabsch, squared-residual inlier count,
    refit on the inliers: ransac.m:40-66 via pcreg_ransac_score), then 10^5 RANSAC-seeded poses (the true pose perturbed as
    good seeds are: <= 6 deg, sigma 1 mm) polished by 20 ICP iterations, 20k source vs 2M model, PLAIN + thDist2 = 4."""
    from pcreg_b200 import synth
    c = C4
    p1, p2, T_true = synth.make_ransac_problem(c["P"], c["inlier_frac"], c["sigma_match"], c["seed"])
    tri = synth.make_triplets(c["P"], c["hyp"], c["seed"] + 1)
    coef = dict(thDist=c["thDist"], thInlrRatio=c["ratio"], REFINE=True, iterNum=c["hyp"])
    P.ransac(p1, p2, coef, triplets=tri[:1000])
    t0 = time.perf_counter()
    for _ in range(steps):
        rr = P.ransac(p1, p2, coef, triplets=tri)
    ransac_ms = (time.perf_counter() - t0) * 1e3 / steps
    model = synth.make_model(c["nm"], c["seed"])
    src, T_gt, ctr = synth.make_source(model, c["ns"], 0.3, c["seed"])
    g = synth.rng(5)
    ang = np.deg2rad(g.uniform(0, 6, c["hyp"]))
    ax = g.standard_normal((c["hyp"], 3))
    tr = g.normal(0, 1.0, (c["hyp"], 3))
    T0 = np.stack([synth.perturb_pose(T_gt, ctr, synth.rot_axis_angle(ax[h], ang[h]), tr[h]) for h in range(c["hyp"])])
    w = dict(nm=c["nm"], ns=c["ns"], hyp=c["hyp"], iters=c["iters"], mode="plain", nn="grid", desc=c["desc"])
    r = gpu_workload(P, torch, w, 0, steps, 1, inputs=(model, src, T0, None, T_gt), opts_kw=dict(thDist2=c["thDist2"]))
    r["roofline"] = roofline_for(w, r)
    sec = r["ms_per_step"] * 1e-3
    return dict(workload=c["desc"], ransac=dict(hypotheses=c["hyp"], pairs=c["P"], ms_per_call=ransac_ms, hyp_per_s=c["hyp"] / (ransac_ms * 1e-3),
                                                max_inliers=int(rr["maxInliers"]), num_success=int(rr["numSuccess"]),
                                                note="host-buffer call: triplet upload + device scoring / refit + result download"),
                polish=dict(value=r["q_per_step"] / sec, unit="queries/s", hyp_per_s=r["H"] / sec, ms_per_step=r["ms_per_step"],
                            e2e=dict(value=r["q_per_step"] / (r["ms_per_step_e2e"] * 1e-3), unit="queries/s", ms_per_step=r["ms_per_step_e2e"],
                                     h2d_bytes_per_step=r["h2d"], d2h_bytes_per_step=r["d2h"], result_equals_device_path=r["e2e_equals_device"]),
                            roofline=r["roofline"], step=step_bytes(w, r), gpu_launches=r["launches"], best_rmse=r["rmse_best"], index=r["grid"],
                            steps=steps, warmup=1),
                total_ms=ransac_ms + r["ms_per_step"], hyp_per_s_end_to_end=c["hyp"] / ((ransac_ms + r["ms_per_step_e2e"]) * 1e-3))


def local_points_workload(P, torch, nk=100_000, nm=16_000_000):
    """Row f2 at the descriptor stage's full size (getSpacialHistogramDescriptors.m:50-60 on the upsampled cloud): 10^5 keypoints
    against a 16 M-point resident model through the C ABI with host buffers.  Models with a grid walk the ball's cell rows;
    the brute-force compaction of grid-less models is timed beside it on 1/50 of the keypoints."""
    from pcreg_b200 import synth, _lib as L
    model = np.asarray(synth.make_model(nm, 1005), dtype=np.float64)
    g = synth.rng(77)
    kp = model[g.integers(0, nm, nk)] + g.normal(0, 0.3, (nk, 3))
    lib = L.lib()

    def count(m, c, R, mn, mx):
        cf = np.asfortranarray(c)
        counts = np.empty(c.shape[0], dtype=np.int64); status = np.empty(c.shape[0], dtype=np.int32)
        a = (m.handle, cf.ctypes.data_as(L.c_f64p), c.shape[0], c.shape[0], R, mn, mx, counts.ctypes.data_as(L.c_i64p), status.ctypes.data_as(L.c_i32p))
        L.check(lib.pcreg_local_points_count(*a), "count")
        t0 = time.perf_counter()
        L.check(lib.pcreg_local_points_count(*a), "count")
        return (time.perf_counter() - t0) * 1e3, counts, status

    def fill(m, c, R, counts, status):
        cf = np.asfortranarray(c)
        off = np.zeros(c.shape[0] + 1, dtype=np.int64)
        np.cumsum(np.where(status == 0, counts, 0), out=off[1:])
        nt = max(int(off[-1]), 1)
        out = np.zeros((nt, 3), dtype=np.float64, order="F"); d = np.zeros(nt); idx = np.zeros(nt, dtype=np.int32)
        a = (m.handle, cf.ctypes.data_as(L.c_f64p), c.shape[0], c.shape[0], R, off.ctypes.data_as(L.c_i64p), status.ctypes.data_as(L.c_i32p),
             out.ctypes.data_as(L.c_f64p), nt, d.ctypes.data_as(L.c_f64p), idx.ctypes.data_as(L.c_i32p))
        L.check(lib.pcreg_local_points_fill(*a), "fill")
        t0 = time.perf_counter()
        L.check(lib.pcreg_local_points_fill(*a), "fill")
        return (time.perf_counter() - t0) * 1e3, out, d, idx, nt

    res = dict(workload="getLocalPoints: %d keypoints x %d-point model, C-ABI calls with host buffers" % (nk, nm))
    mg = P.Model(model, grid=True, voxel_map=-1)
    ms, cnt, st = count(mg, kp, 3.5, 30, 6000)
    res["count_R3.5"] = dict(ms=ms, keypoints=nk, mean_points_in_ball=float(cnt.mean()), accepted=int((st == 0).sum()),
                             note="getSpacialHistogramDescriptors.m's options on this density: every ball exceeds max_pts = 6000")
    ms, cnt, st = count(mg, kp, 1.2, 30, 6000)
    res["count_R1.2"] = dict(ms=ms, keypoints=nk, mean_points_in_ball=float(cnt.mean()), accepted=int((st == 0).sum()))
    sub = kp[::10]
    cs, ss = cnt[::10].copy(), st[::10].copy()
    ms, o1, d1, i1, nt = fill(mg, sub, 1.2, cs, ss)
    res["fill_R1.2"] = dict(ms=ms, keypoints=int(sub.shape[0]), points_out=nt, d2h_bytes=nt * 36,
                            note="the call is its device-to-host copy: 36 B per neighbourhood point into pageable host arrays")
    mb = P.Model(model)
    few = kp[::50]
    msb, cb, sb = count(mb, few, 1.2, 30, 6000)
    res["brute_count_R1.2"] = dict(ms=msb, keypoints=int(few.shape[0]), note="grid-less model: order-preserving brute-force compaction")
    ms2, o2, d2, i2, nt2 = fill(mb, sub[::5], 1.2, cb, sb)
    sel = np.concatenate([[0], np.cumsum(np.where(ss == 0, cs, 0))])
    rows = np.concatenate([np.arange(sel[k], sel[k + 1]) for k in range(0, sub.shape[0], 5)]) if nt2 > 1 else np.arange(0)
    res["grid_equals_brute"] = bool(np.array_equal(cb, cnt[::50]) and np.array_equal(o1[rows], o2[:rows.size]) and np.array_equal(d1[rows], d2[:rows.size])
                                    and np.array_equal(i1[rows], i2[:rows.size]))
    mg.destroy(); mb.destroy()
    return res


def side_leg(line, key, fn):
    t0 = time.perf_counter()
    try:
        line[key] = fn()
        if isinstance(line[key], dict):
            line[key]["leg_seconds"] = round(time.perf_counter() - t0, 1)
    except Exception as e:                                                       # a side leg never takes the headline down
        line[key] = dict(error="%s: %s" % (type(e).__name__, e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    for name, what in (("c2", "C2 (brute-force) measurement"), ("cpu", "cpu_baseline leg"), ("match", "getMatches (row f4) measurement"),
                       ("c4", "C4 (RANSAC-seeded refinement) leg"), ("c5", "C5 (16M-point model) leg"), ("align", "AlignPoints-batch leg"),
                       ("local", "getLocalPoints (row f2) leg"), ("strong", "strong-scaling leg at N > 1"), ("e2e-multi", "single-process multi-device e2e leg at N > 1")):
        ap.add_argument("--no-" + name, action="store_true", help="skip the " + what)
    ap.add_argument("--only", action="store_true", help="headline only (all side legs off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the headline's last timed step returned (rank 0's share at N > 1) "
                         "as DIR/<name>.npy in float64, to compare two builds output for output on the same seeded inputs")
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    off = lambda n: args.only or getattr(args, "no_" + n.replace("-", "_"))

    if args.impl == "reference":
        run_reference(args, w, rank, world)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = hostpg = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        hostpg = dist.new_group(backend="gloo")              # host-side barrier: the waiting ranks must not spin on their GPUs
    import pcreg_b200 as P
    P.init(local_rank)
    warmup = max(3, args.warmup)

    r = gpu_workload(P, torch, w, rank, args.steps, warmup, dist, world, do_e2e=(world == 1), keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in r["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    r["roofline"] = roofline_for(w, r)
    sec = r["ms_per_step"] * 1e-3
    value = r["q_per_step"] * world / sec
    line = dict(metric="ICP NN queries/s", value=value, unit="queries/s", n_gpus=world, steps=args.steps, warmup=warmup,
                ms_per_step=r["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=config_of(w, r["H"], world), hyp_per_s=r["H"] * world / sec,
                gpu_launches=r["launches"], clocks=r["clocks"], ms_per_step_by_rank=r["ms_ranks"], per_step_ms=r["per_step_ms"],
                roofline=r["roofline"], step=step_bytes(w, r), index=r["grid"],
                kernel_time_share=dict(nn_ms=r["prof_t"]["nn_ms"], update_ms=r["prof_t"]["update_ms"], list_ms=r["prof_t"]["list_ms"],
                                       rowscan_ms=r["prof_t"]["rowscan_ms"], walk_ms=r["prof_t"]["walk_ms"], step_ms=r["ms_per_step"],
                                       fused=bool(r["prof"].get("fused")),
                                       note="CUDA-event times from one extra profiled step without counters, not from the timed steps"),
                best_rmse=r["rmse_best"])
    if world == 1:
        line["e2e"] = dict(value=r["q_per_step"] / (r["ms_per_step_e2e"] * 1e-3), unit="queries/s", h2d_bytes_per_step=r["h2d"],
                           d2h_bytes_per_step=r["d2h"], ms_per_step=r["ms_per_step_e2e"], hyp_per_s=r["H"] / (r["ms_per_step_e2e"] * 1e-3),
                           result_equals_device_path=r["e2e_equals_device"])
    # ---- strong scaling: BASELINE.json's config 3 as stated (4096 poses in total) ----
    if world > 1 and not off("strong") and args.workload == "c3":
        model_h, src, T0_all, w_src, T_gt = make_inputs(w, 0, 1)
        rs = gpu_workload(P, torch, w, rank, args.steps, 2, dist, world, T0_override=np.ascontiguousarray(T0_all[rank::world]),
                          do_e2e=False, do_profile=False, inputs=(model_h, src, T0_all, w_src, T_gt))
        t1 = r["ms_per_step"]                                  # 4096 poses on ONE GPU: what every rank just did in the weak run
        line["strong"] = dict(hypotheses_total=int(T0_all.shape[0]), hypotheses_per_gpu=rs["H"], ms_per_step=rs["ms_per_step"],
                              value=rs["q_per_step"] * world / (rs["ms_per_step"] * 1e-3), unit="queries/s",
                              efficiency=t1 / (world * rs["ms_per_step"]), gpu_launches=rs["launches"], ms_per_step_by_rank=rs["ms_ranks"],
                              note="efficiency = (ms per step of 4096 poses on one GPU, this run's weak-scaling step) / (N x ms per step of "
                                   "4096 / N poses per GPU); includes the all-gather of records, the arg-min and the 8-byte result read")
    # ---- e2e at N > 1: one process, all devices, through the C ABI ----
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=hostpg)
        if rank == 0 and not off("e2e-multi"):
            try:
                e = e2e_multi_device(P, torch, w, world, args.steps)
                line["e2e"] = dict(value=e["H"] * w["ns"] * (w["iters"] + 1) / (e["ms_per_step_e2e"] * 1e-3), unit="queries/s",
                                   h2d_bytes_per_step=e["h2d"], d2h_bytes_per_step=e["d2h"], ms_per_step=e["ms_per_step_e2e"],
                                   hyp_per_s=e["H"] / (e["ms_per_step_e2e"] * 1e-3), best_rmse=e["rmse_best"], how=e["how"])
            except Exception as ex:
                line["e2e"] = dict(error="%s: %s" % (type(ex).__name__, ex))
        dist.barrier(group=hostpg)
    # ---- the other configurations, N = 1 only ----
    if rank == 0 and world == 1 and args.workload == "c3":
        if not off("c2"):
            def c2_leg():
                w2 = WORKLOADS["c2"]
                r2 = gpu_workload(P, torch, w2, 0, max(2, args.steps), 3)
                r2["roofline"] = roofline_for(w2, r2)
                s2 = r2["ms_per_step"] * 1e-3
                d = dict(workload=w2["desc"], value=r2["q_per_step"] / s2, unit="queries/s", ms_per_step=r2["ms_per_step"], hyp_per_s=1.0 / s2,
                         e2e=dict(value=r2["q_per_step"] / (r2["ms_per_step_e2e"] * 1e-3), unit="queries/s", ms_per_step=r2["ms_per_step_e2e"]),
                         roofline=r2["roofline"], gpu_launches=r2["launches"], best_rmse=r2["rmse_best"], clocks=r2["clocks"])
                w3 = WORKLOADS["c2g"]
                r3 = gpu_workload(P, torch, w3, 0, max(2, args.steps), 3)
                d["grid_path"] = dict(workload=w3["desc"], value=r3["q_per_step"] / (r3["ms_per_step"] * 1e-3), unit="queries/s",
                                      ms_per_step=r3["ms_per_step"], e2e_ms_per_step=r3["ms_per_step_e2e"], best_rmse=r3["rmse_best"],
                                      gpu_launches=r3["launches"], same_result_as_brute=bool(r3["rmse_best"] == r2["rmse_best"]))
                return d
            side_leg(line, "c2", c2_leg)
        if not off("match"):
            side_leg(line, "get_matches", lambda: match_workload(P, torch))
        if not off("align"):
            side_leg(line, "align_batch", lambda: align_batch_workload(P, torch))
        if not off("c4"):
            side_leg(line, "c4", lambda: c4_workload(P, torch))
        if not off("local"):
            side_leg(line, "local_points", lambda: local_points_workload(P, torch))
        if not off("c5"):
            def c5_leg():
                w5 = WORKLOADS["c5"]
                r5 = gpu_workload(P, torch, w5, 0, 2, 1)
                r5["roofline"] = roofline_for(w5, r5)
                s5 = r5["ms_per_step"] * 1e-3
                return dict(workload=w5["desc"], value=r5["q_per_step"] / s5, unit="queries/s", hyp_per_s=r5["H"] / s5, ms_per_step=r5["ms_per_step"],
                            steps=2, warmup=1, e2e=dict(value=r5["q_per_step"] / (r5["ms_per_step_e2e"] * 1e-3), unit="queries/s",
                                                        ms_per_step=r5["ms_per_step_e2e"], h2d_bytes_per_step=r5["h2d"], d2h_bytes_per_step=r5["d2h"]),
                            roofline=r5["roofline"], step=step_bytes(w5, r5), gpu_launches=r5["launches"], best_rmse=r5["rmse_best"], index=r5["grid"],
                            note="one GPU's share of configs[4] (16 384 hypotheses over 8 GPUs); the model is not L2-resident: DRAM bytes = algorithmic bytes")
            side_leg(line, "c5", c5_leg)
    if rank == 0 and world == 1 and not off("cpu"):
        cores = os.cpu_count() or 1
        c = cpu_sample(w, budget_s=15.0)
        line["cpu_baseline"] = dict(value=c["queries_per_s"], unit="queries/s", cores=cores, kind="port",
                                    hyp_per_s=c["hyp_per_s"],
                                    sample="%d of the %d hypotheses of the same workload, full %d iterations each (%.1f s; oracle restatement: "
                                           "numpy FP64 + scipy cKDTree workers=-1, tree build %.1f s excluded; MATLAB/Octave %s)"
                                           % (c["n_hyp"], r["H"], w["iters"], c["seconds"], c["kdtree_build_s"],
                                              "not installed" if not probe_matlab() else "present: " + ",".join(probe_matlab())))
    if world > 1:
        dist.barrier(group=hostpg)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
