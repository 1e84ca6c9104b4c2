#!/usr/bin/env python
"""bench.py - forward+backward throughput of the rasterizer hot path (BASELINE.json metric:
"fwd+bwd Mpix/s @1M Gaussians/1024^2; HBM GB/s vs roofline; 1/2/4/8 GPU").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one view of the workload rendered (forward) and back-propagated (backward) through
the public drop-in API (GaussianRasterizer -> C ABI -> sm_100a kernels).  N>1 (torchrun, one
rank per GPU): every rank renders its own view of the replicated scene (weak scaling: 1 view per
GPU, SURVEY.md 8e) and the parameter gradients are all-reduced over NCCL inside backward.

Prints ONE JSON line (rank 0).  See the task contract for the keys; additions:
  roofline      dominant kernel's algorithmic bytes / its measured launch time vs measured HBM peak
  cpu_baseline  the pure-PyTorch CPU oracle timed on this box on a bounded sample (N=1 only)
  stages_ms     mean device time of every kernel stage over the timed steps
--impl reference times the CPU oracle port (the reference's CUDA op is un-vendored; DESIGN.md).
--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (rank 0;
see dump_sample), so that two builds can be compared output for output on identical inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from harness import cameras, synthetic  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[2]: 1M Gaussians, 1024x1024 (object-like ball R=0.5) - the metric's config.
    # Scales follow the reference recipe exactly (3-NN distances, gs_renderer.py:590-594; SURVEY 8d):
    # D ~ 4.8M tile pairs.  Round 1 benchmarked the analytic stand-in for the 3-NN distance (D = 6.38M);
    # that workload stays available as cfg3_r1scales for round-to-round comparisons.
    "cfg3_1M_1024": dict(P=1_000_000, H=1024, W=1024, radius=0.5, opacity="sigmoid_normal"),
    "cfg3_r1scales": dict(P=1_000_000, H=1024, W=1024, radius=0.5, opacity="sigmoid_normal", exact_knn=False),
    "cfg3b_1M_1024_screenfill": dict(P=1_000_000, H=1024, W=1024, radius=1.5, opacity="sigmoid_normal"),
    "cfg2_100k_512": dict(P=100_000, H=512, W=512, radius=0.5, opacity="sigmoid_normal"),
    "cfg2b_81920_512": dict(P=81_920, H=512, W=512, radius=0.5, opacity="sigmoid_normal"),
    "cfg1_10k_256": dict(P=10_000, H=256, W=256, radius=0.5, opacity="sigmoid_normal"),
}
METRIC = "fwd+bwd Mpix/s @1M Gaussians/1024^2"
KERNELS_PER_STEP = 9   # project_sh, multisplit<count>, scan_order, multisplit<scatter>, sort_big, sort_small, composite_fwd, composite_bwd, project_bwd


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_scene(wl, view, device=None):
    sc = synthetic.ball_scene(wl["P"], radius=wl["radius"], sh_degree_max=3, seed=0, opacity=wl["opacity"],
                              exact_knn=wl.get("exact_knn", True))
    cam = cameras.orbit_camera(radius=3.5, theta_deg=60.0, phi_deg=45.0 * view, fovx=0.55,
                               height=wl["H"], width=wl["W"])
    g = torch.Generator().manual_seed(100 + view)
    n = wl["H"] * wl["W"]
    gc = torch.randn(3, wl["H"], wl["W"], generator=g) / n
    gd = torch.randn(2, wl["H"], wl["W"], generator=g) / n
    return sc, cam, gc, gd


# ---------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi in the background during the timed regions)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.path = gpu_index, None, None

    def start(self):
        if os.environ.get("BENCH_NO_CLOCKS"):       # diagnostics only: does the sampler perturb the run?
            return
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # median over the samples taken under load (power above the idle floor)
        thr = min(power) + 0.3 * (max(power) - min(power))
        load = [s for s, p in zip(sm, power) if p >= thr] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(power))}


# ---------------------------------------------------------------------------------------------
# CPU baseline: the oracle (kind "port") on a bounded sample of the same workload
# ---------------------------------------------------------------------------------------------
def cpu_oracle_step(wl, view, sample_stride=8, threads=None, scene=None, group=8):
    """One bounded CPU step: the per-Gaussian stages (fwd+bwd) on all P Gaussians + blending fwd+bwd on
    every `sample_stride`-th non-empty tile (ordered by list length, so the sample spans the length
    distribution; 1/8 = 12.5% of the tiles), extrapolated to the full frame by (tile, Gaussian)-pair
    count.  Tiles are blended in small groups so autograd holds a few tiles' intermediates at a time."""
    from oracle import splat_ref as O
    # all host cores up to 32: beyond that PyTorch's intra-op pool only adds contention for these
    # op sizes (measured on the 128-core box: 128 threads 5127 s/step vs 32 threads far less)
    threads = threads or int(os.environ.get("BENCH_CPU_THREADS", min(os.cpu_count() or 1, 32)))
    torch.set_num_threads(threads)
    sc, cam, gc, gd = scene if scene is not None else make_scene(wl, view)
    S = O.Settings(cam.image_height, cam.image_width, cam.tanfovx, cam.tanfovy, torch.ones(3), 1.0,
                   cam.world_view_transform, cam.full_proj_transform, 3, cam.camera_center, False, False)
    t = {k: v.clone().requires_grad_(True) for k, v in sc.items()}
    m2d = torch.zeros(wl["P"], 3, requires_grad=True)
    t0 = time.perf_counter()
    pre = O.preprocess(S, t["means3D"], t["opacities"], shs=t["shs"], scales=t["scales"],
                       rotations=t["rotations"], means2D=m2d)
    t1 = time.perf_counter()
    _, pl, ranges = O.bin_and_sort(pre, S)
    t2 = time.perf_counter()
    n = ranges[:, 1] - ranges[:, 0]
    order = np.argsort(-n, kind="stable")
    nonempty = int((n > 0).sum())
    tiles = [int(x) for x in order[:max(nonempty, 1):sample_stride]]
    pairs_total, pairs_sample = int(n.sum()), int(n[tiles].sum())
    # leaves between the two stages so their backward passes can be timed separately
    keys = ["px", "py", "opacity", "rgb", "depth"]
    mid = {k: pre[k].detach().requires_grad_(True) for k in keys}
    con = [c.detach().requires_grad_(True) for c in pre["conic"]]
    pre2 = dict(pre); pre2.update(mid); pre2["conic"] = tuple(con)
    leaves = [mid[k] for k in keys] + con
    acc = [torch.zeros_like(x) for x in leaves]
    t3 = time.perf_counter()
    for i in range(0, len(tiles), group):
        color, da, _, _ = O.composite(pre2, pl, ranges, S, tiles=tiles[i:i + group])
        loss = (color * gc).sum() + (da * gd).sum()
        for a, g in zip(acc, torch.autograd.grad(loss, leaves, allow_unused=True)):
            if g is not None:
                a += g
    t5 = time.perf_counter()
    outs = [pre[k] for k in keys] + list(pre["conic"])
    pairs = [(o, g) for o, g in zip(outs, acc) if o.requires_grad]
    torch.autograd.backward([o for o, _ in pairs], [g for _, g in pairs])
    t6 = time.perf_counter()
    per_gauss = (t1 - t0) + (t2 - t1) + (t6 - t5)
    blend = t5 - t3
    scale = pairs_total / max(pairs_sample, 1)
    est_full = per_gauss + blend * scale
    return dict(est_full_s=est_full, wall_s=t6 - t0, per_gaussian_s=per_gauss, blend_sample_s=blend,
                pairs_total=pairs_total, pairs_sample=pairs_sample, tiles_sampled=len(tiles),
                tiles_nonempty=nonempty, threads=threads, sample_stride=sample_stride)


def cpu_baseline_dict(wl, r, spread=None):
    mpix = wl["H"] * wl["W"] / r["est_full_s"] / 1e6
    d = {"value": mpix, "unit": "Mpix/s", "cores": r["threads"], "kind": "port",
         "sample": (f"oracle/splat_ref.py (pure PyTorch fp32, {r['threads']} threads): per-Gaussian stages "
                    f"fwd+bwd on all {wl['P']} Gaussians ({r['per_gaussian_s']:.2f}s) + blending fwd+bwd on "
                    f"{r['tiles_sampled']} of {r['tiles_nonempty']} non-empty tiles (every {r['sample_stride']}th by list "
                    f"length, {r['pairs_sample']} of {r['pairs_total']} pairs = {100.0 * r['pairs_sample'] / max(r['pairs_total'], 1):.1f}%, "
                    f"{r['blend_sample_s']:.2f}s) scaled by pair count -> {r['est_full_s']:.1f}s per full step")}
    if spread:
        d["spread"] = spread
    return d


# ---------------------------------------------------------------------------------------------
def run_reference(args, wl_name, wl, rank, world):
    """--impl reference: the CPU oracle port on the host cores (the reference's CUDA op is un-vendored
    and its own CPU path does not exist).  One "step" is the bounded sample of cpu_oracle_step;
    ms_per_step is that sample's wall time (so steps x ms_per_step is what the run really took) and
    `value` is the throughput of the full workload extrapolated from it."""
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    res = []
    scene = make_scene(wl, 0)     # synthetic inputs are built once, outside the timed steps
    for i in range(warm + steps):
        r = cpu_oracle_step(wl, 0, scene=scene)
        if i >= warm:
            res.append(r)
    est_all = np.array([r["est_full_s"] for r in res])
    est = float(np.median(est_all))
    wall = float(np.mean([r["wall_s"] for r in res]))
    r0 = dict(res[-1]); r0["est_full_s"] = est
    mp = wl["H"] * wl["W"] / est_all / 1e6
    cb = cpu_baseline_dict(wl, r0, spread={"steps": len(res), "min": float(mp.min()), "median": float(np.median(mp)),
                                           "max": float(mp.max())})
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "Mpix/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": wall * 1e3, "full_step_ms_extrapolated": est * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(wl_name, wl, world),
            "note": ("reference CUDA op is un-vendored: CPU oracle port timed. ms_per_step = wall time of one bounded "
                     "sample step; value = full-frame throughput extrapolated from it by pair count"),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_ROWS = 1 << 16                  # per-Gaussian outputs are sampled: 1M full rows would be ~250 MB
DUMP_MAX_BYTES = 64 << 20


def dump_sample(color, radii, da, grads, P):
    """Host copy of one step's results as its caller receives them: the rendered colour [3,H,W] and
    depth/alpha [2,H,W] in full; radii and the gradients of every input on DUMP_ROWS Gaussians drawn
    with a fixed seed (their indices are written as sample_index).  All float32 or float64."""
    idx = np.sort(np.random.RandomState(0).choice(P, min(P, DUMP_ROWS), replace=False))
    sel = torch.from_numpy(idx).to(color.device)
    out = {"color": color, "depth_alpha": da, "radii": radii.index_select(0, sel).float()}
    out.update({f"grad_{k}": g.index_select(0, sel) for k, g in grads.items()})
    out = {k: v.detach().cpu().numpy() for k, v in out.items()}
    out["sample_index"] = idx.astype(np.float64)
    assert sum(v.nbytes for v in out.values()) <= DUMP_MAX_BYTES
    return out


def workload_config(wl_name, wl, world, sh_degree=3):
    """The `config` object both arms print (identical keys, so the driver sees the same config)."""
    return {"workload": wl_name, "P": wl["P"], "H": wl["H"], "W": wl["W"], "sh_degree": sh_degree, "M": 16,
            "views_per_step": world, "parallelism": f"view-sharded dp{world}",
            "scales": "exact 3-NN (reference recipe)" if wl.get("exact_knn", True) else "analytic 3-NN stand-in (round-1 workload)"}


def secondary_roofline(evals, mean_ms, clk):
    """SURVEY 8(d) secondary roofline: what actually bounds the composite kernels once records sit in
    shared memory is the rate of (pixel, Gaussian) evaluations (each warp-level pair = 32 of them,
    ~20 fp32 ops + 1 MUFU.EX2 in the forward, ~60 + 2 MUFU in the backward), against the SM's issue
    peaks at the measured clock: 4 warp-instructions/clk/SM issue, 16 MUFU lanes/clk/SM."""
    mhz = (clk or {}).get("sm_mhz") or 1965.0
    sms = 148
    issue_peak = sms * 4 * mhz * 1e6                    # warp instructions / s
    mufu_peak = sms * 16 * mhz * 1e6                    # lane-level ex2/rcp per s
    out = {"unit": "pixel-pair evaluations/s", "sm_mhz": mhz, "counts": evals,
           "mufu_peak_lanes_per_s": mufu_peak, "issue_peak_warp_instr_per_s": issue_peak}
    for name, key, mufu_per_eval in (("composite_fwd", "fwd_pairs_evaluated", 1), ("composite_bwd", "bwd_pairs_evaluated", 1)):
        t = mean_ms.get(name)
        n = evals.get(key, 0)
        if t and n:
            rate = 32.0 * n / (t * 1e-3)
            out[name] = {"evals_per_s": rate, "frac_of_mufu_peak": rate * mufu_per_eval / mufu_peak,
                         "issue_slots_per_warp_pair": issue_peak * t * 1e-3 / n}
    return out


def algorithmic_bytes(P, V, D, N, M):
    """Minimum-traffic model per kernel (SURVEY.md 8d mapped onto this design; DESIGN.md)."""
    g_in = 44 + 12 * M
    return {
        "project_sh": P * g_in + P * (4 + 16) + V * 48,        # params; radii + rect/depth; geom record
        "scan_order": 0,
        "scatter": P * 16 + D * 8,                               # rect/depth read; key write
        "tile_sort": D * 8 * 2,                                  # key read + sorted key write
        "composite_fwd": D * (8 + 48) + N * (12 + 8 + 4),        # keys + gathered records; colour, depth_alpha, n_contrib
        "composite_bwd": D * (8 + 48) + N * (20 + 8) + V * 48,   # keys + records; grads in + T/n_contrib; dgeom
        "project_bwd": P * g_in + V * 48 + P * 4 + P * (g_in + 12),  # params, dgeom, radii; grads out
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3_1M_1024", choices=sorted(WORKLOADS))
    ap.add_argument("--sh-degree", type=int, default=3, help="active SH degree (the metric's config is 3)")
    ap.add_argument("--reduce", default="backward", choices=["backward", "deferred"],
                    help="N>1: chunk-overlapped all-reduce inside the rasterizer backward, or DDP-style "
                         "all-reduce of the leaf gradients after it (dreamscene_b200.parallel)")
    ap.add_argument("--sh-exchange", default="factored", choices=["factored", "dense"],
                    help="N>1, --reduce backward: SH gradient exchanged as [P,3] colour gradients + camera centre "
                         "(all-gather, rebuilt locally) or all-reduced as [P,M,3] rows")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    wl_name, wl = args.workload, WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, wl_name, wl, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    from dreamscene_b200 import GaussianRasterizationSettings, GaussianRasterizer, _lib, parallel
    from dreamscene_b200 import rasterizer as R
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback in the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        parallel.enable_view_sharding(mode=args.reduce, sh_exchange=args.sh_exchange)
    _lib.load()

    sc, cam, gc_h, gd_h = make_scene(wl, rank)
    P, H, W, M = wl["P"], wl["H"], wl["W"], 16
    names = ("means3D", "opacities", "shs", "scales", "rotations")
    host = {k: sc[k].pin_memory() for k in names}
    prm = {k: host[k].to(dev).requires_grad_(True) for k in names}
    gc, gd = gc_h.to(dev), gd_h.to(dev)
    S = GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
        bg=torch.ones(3, device=dev), scale_modifier=1.0, viewmatrix=cam.world_view_transform.to(dev),
        projmatrix=cam.full_proj_transform.to(dev), sh_degree=args.sh_degree, campos=cam.camera_center.to(dev),
        prefiltered=False, score_flag=False)
    rast = GaussianRasterizer(S)
    m2d = torch.zeros(P, 3, device=dev, requires_grad=True)

    def step(p):
        for v in p.values():
            v.grad = None
        m2d.grad = None
        color, radii, da = rast(means3D=p["means3D"], means2D=m2d, opacities=p["opacities"], shs=p["shs"],
                                scales=p["scales"], rotations=p["rotations"])
        torch.autograd.backward([color, da], [gc, gd])
        if world > 1 and args.reduce == "deferred":
            parallel.all_reduce_gradients(list(p.values()), active_columns={p["shs"]: (args.sh_degree + 1) ** 2})
        return color, radii, da

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # nvidia-smi takes a driver-wide lock for tens of ms while it initialises: start the sampler
    # BEFORE the warm-up so that stall never lands inside the timed region (it did in the first
    # round-2 run: one 76 ms step)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(1.0)
    for _ in range(args.warmup):
        color, radii, da = step(prm)
    barrier()
    V = int((radii > 0).sum())
    D = int(R.last_pair_count(dev))

    # pair-evaluation counts for the secondary roofline: ONE extra, untimed step with the
    # instrumented kernel instantiations
    counters = torch.zeros(_lib.STAT_WORDS, dtype=torch.int64, device=dev)
    _lib.debug_counters(counters.data_ptr())
    step(prm)
    torch.cuda.synchronize(dev)
    _lib.debug_counters(None)
    evals = {k: int(x) for k, x in zip(_lib.STAT_NAMES, counters.tolist()) if not k.startswith("_")}
    balance = {}
    for side in ("fwd", "bwd"):      # load balance of the persistent kernels (instrumented instantiation, untimed)
        span = evals.pop(f"{side}_end_ns") - ~evals.pop(f"{side}_not_begin_ns")   # the word holds ~begin (atomicMax = min)
        busy, workers = evals.pop(f"{side}_busy_ns"), evals.pop(f"{side}_workers")
        balance[side] = {"workers": workers, "span_us": span / 1e3,
                         "mean_busy_frac": busy / max(1, workers * span),
                         "longest_item_us": evals.pop(f"{side}_max_item_ns") / 1e3}
    balance["bwd"]["most_evals_in_one_item"] = evals.pop("bwd_max_item_evals")

    # ---- timed region 1: device-resident inputs --------------------------------------------
    _lib.profile_enable(args.steps)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]   # per-step spread only
    barrier()
    e0.record()
    marks[0].record()
    for i in range(args.steps):
        color, radii, da = step(prm)
        marks[i + 1].record()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    per_step = np.array([marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)])
    stages = _lib.profile_collect()
    _lib.profile_enable(0)
    R.flush_checks(dev)             # every forward's pair count has been checked against its capacity
    dump = None
    if args.dump_outputs and rank == 0:     # before grad_check and e2e overwrite the gradients
        dump = dump_sample(color, radii, da, {**{k: prm[k].grad for k in names}, "means2D": m2d.grad}, P)
    t_ms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_step = float(t_ms.item()) / args.steps
    value = world * H * W / (ms_step * 1e-3) / 1e6

    # ---- multi-GPU correctness: the reduced gradient of the sharded step == the sum over all views
    # rendered sequentially on this one GPU (what DreamScene's loop computes) ------------------------
    grad_check = None
    if world > 1:
        step(prm)
        reduced = torch.cat([prm[k].grad.reshape(-1) for k in names]).clone()
        parallel.disable_view_sharding()
        reduce_mode, args.reduce = args.reduce, "none"
        total = torch.zeros_like(reduced)
        for v in range(world):
            sc_v, cam_v, gc_v, gd_v = make_scene(wl, v) if v != rank else (sc, cam, gc_h, gd_h)
            S_v = S._replace(viewmatrix=cam_v.world_view_transform.to(dev), projmatrix=cam_v.full_proj_transform.to(dev),
                             campos=cam_v.camera_center.to(dev))
            for t_ in prm.values():
                t_.grad = None
            c_, _, a_ = GaussianRasterizer(S_v)(means3D=prm["means3D"], means2D=m2d, opacities=prm["opacities"],
                                                shs=prm["shs"], scales=prm["scales"], rotations=prm["rotations"])
            torch.autograd.backward([c_, a_], [gc_v.to(dev), gd_v.to(dev)])
            total += torch.cat([prm[k].grad.reshape(-1) for k in names])
        args.reduce = reduce_mode
        parallel.enable_view_sharding(mode=args.reduce, sh_exchange=args.sh_exchange)
        err = ((reduced - total).double().norm() / total.double().norm().clamp_min(1e-300)).reshape(1)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        grad_check = {"rel_err_max_over_ranks": float(err.item()), "views_summed": world,
                      "what": "all-reduced parameter gradients vs the sum of all views' gradients recomputed on each rank"}
        barrier()

    # ---- timed region 2: end to end with HOST buffers (H2D inputs, D2H results every step) --
    e2e = None
    if not args.no_e2e:
        out_host = {"color": torch.empty(3, H, W).pin_memory(), "da": torch.empty(2, H, W).pin_memory(),
                    "radii": torch.empty(P, dtype=torch.int32).pin_memory()}
        grad_host = {k: torch.empty_like(host[k]).pin_memory() for k in names}
        h2d = sum(host[k].numel() * 4 for k in names) + (16 + 16 + 3 + 3) * 4
        d2h = sum(v.numel() * 4 for v in out_host.values()) + sum(v.numel() * 4 for v in grad_host.values())

        NS = 3   # steps in flight: H2D of step i+1/i+2 overlaps compute and D2H of step i (full-duplex PCIe)
        streams = [torch.cuda.Stream(dev) for _ in range(NS)]
        outs = [dict(out_host)] + [{k: torch.empty_like(v).pin_memory() for k, v in out_host.items()} for _ in range(NS - 1)]
        gouts = [dict(grad_host)] + [{k: torch.empty_like(v).pin_memory() for k, v in grad_host.items()} for _ in range(NS - 1)]

        def e2e_step(i):
            # every step: H2D of all inputs from pinned memory, forward+backward through the public
            # API, D2H of the rendered maps and of every parameter gradient.  Steps rotate over NS
            # streams so one step's D2H overlaps the next steps' H2D; a stream is only reused after
            # its previous step has fully completed (host results owned by the caller).
            st = streams[i % NS]
            st.synchronize()
            with torch.cuda.stream(st):
                p = {k: host[k].to(dev, non_blocking=True).requires_grad_(True) for k in names}
                color, radii_, da = step(p)
                oh, gh = outs[i % NS], gouts[i % NS]
                oh["color"].copy_(color.detach(), non_blocking=True)
                oh["da"].copy_(da.detach(), non_blocking=True)
                oh["radii"].copy_(radii_, non_blocking=True)
                for k in names:
                    gh[k].copy_(p[k].grad, non_blocking=True)

        for i in range(NS):
            e2e_step(i)
        for st in streams:
            st.synchronize()
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            e2e_step(i)
        for st in streams:
            st.synchronize()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_ms = float(dt.item()) * 1e3 / args.steps
        e2e = {"value": world * H * W / (e2e_ms * 1e-3) / 1e6, "unit": "Mpix/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "note": "3 steps in flight on 3 streams: D2H of step i overlaps H2D of steps i+1, i+2"}
    clk = clocks.stop() if rank == 0 else None

    if rank == 0:
        peak, peak_src = measured_peaks()
        alg = algorithmic_bytes(P, V, D, H * W, M)
        mean_ms = {k: float(np.mean(v)) for k, v in stages.items() if v}
        dom = max(mean_ms, key=mean_ms.get)
        achieved = alg[dom] / (mean_ms[dom] * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get(wl_name, {}).get(dom)
            except Exception:
                traffic = None
        step_alg = sum(alg.values())
        line = {
            "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(wl_name, wl, world, args.sh_degree),
            "workload_stats": {"visible": V, "tile_pairs": D,
                               "l2": "inputs larger than L2 (params 236 MB read + 248 MB grads written + %d MB keys per step)" % (D * 8 // 2**20)},
            "ms_per_step_spread": {"median": float(np.median(per_step)), "min": float(per_step.min()),
                                   "max": float(per_step.max())},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg[dom], "ms_per_launch": mean_ms[dom],
                         "secondary": secondary_roofline(evals, mean_ms, clk), "load_balance": balance},
            "step_hbm": {"algorithmic_bytes": step_alg, "achieved_gbs": step_alg / (ms_step * 1e-3) / 1e9,
                         "frac": step_alg / (ms_step * 1e-3) / 1e9 / peak},
            "stages_ms": mean_ms,
            "clocks": clk,
            "gpu_launches": KERNELS_PER_STEP * args.steps,
        }
        if e2e:
            line["e2e"] = e2e
        if grad_check:
            line["grad_check"] = grad_check
            ncoef = (args.sh_degree + 1) ** 2
            floats = 3 + 1 + 3 * ncoef + 3 + 4
            if args.reduce == "backward" and args.sh_exchange == "factored":
                line["limiting_collective"] = (
                    f"inside backward: ncclAllGather of [P,3] colour gradients + camera centre ({12 * P / 1e6:.0f} MB sent, "
                    f"{12 * P * world / 1e6:.0f} MB received per rank; the [P,M,3] SH gradient is rebuilt locally by "
                    f"sh_grad_expand) + ncclAllReduce(SUM, fp32) of the other parameter gradients (11 floats/Gaussian = "
                    f"{44 * P / 1e6:.0f} MB)")
            else:
                line["limiting_collective"] = (
                    f"ncclAllReduce(SUM, fp32) of the parameter gradients: {floats} floats/Gaussian = {floats * 4 * P / 1e6:.0f} MB/step "
                    + ("one call on the rasterizer's flat gradient buffer, inside backward" if args.reduce == "backward"
                       else "one call on the flattened leaf gradients after backward (DDP-style)"))
            line["reduce_mode"] = args.reduce if args.reduce != "backward" else f"backward/{args.sh_exchange}"
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_dict(wl, cpu_oracle_step(wl, 0))
        if dump:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for k, v in dump.items():
                np.save(os.path.join(args.dump_outputs, f"{k}.npy"), v)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
