#!/usr/bin/env python
"""bench.py -- training views/sec (fwd + bwd + Adam) of the B200-native 3DGS rasterizer.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one batch of synthetic views: every view is rendered (projection +
SH + tile sort + blend forward), its L1 + fused-SSIM photometric gradient (the reference's loss) is back-propagated (blend backward + per-Gaussian
backward), gradients of the batch are summed (NCCL all-reduce across ranks) and ONE fused Adam step is taken.
Workload = BASELINE.json configs[2] ("C3": 1M Gaussians, 8 views of 1920x1080 per GPU, SH degree 3); with N GPUs
the global batch is 8 N views (weak scaling; the views of a step are sharded round-robin over the ranks).

One JSON line is printed by rank 0 (see the contract in the task statement): `value` = views/s with the target
images already resident in HBM; `e2e` = the same through SplatTrainer.train_step with pinned HOST uint8 targets
(H2D per view, D2H of the loss per step); `roofline` = blend-backward kernel, algorithmic bytes (172 I + 24 P per
view, BASELINE.md section 5) over its CUDA-event time against MEASURED_PEAKS.json; `cpu_baseline` = the CPU oracle
port timed on whole views of the same workload (bounded sample: one to three views); `reference_gpu` = the reference's
own training step (its autograd Functions, fused SSIM and FusedAdam, compiled unchanged) on its own CUDA backends, timed
in child processes beside ours.  --config C4 = 32 views with the mcmc regularisers; --scaling strong = fixed total views.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "training views/sec (fwd+bwd+Adam) @1M Gaussians 1080p"
UNIT = "views/s"
LAMBDA_DSSIM = 0.2  # eval/default_optimization_params.json; loss = (1-l) L1 + l (1 - SSIM), src/training/trainer.cpp:122-125


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3")
    ap.add_argument("--n-gaussians", type=int, default=0, help="override N (testing only; invalidates the metric)")
    ap.add_argument("--views-per-gpu", type=int, default=0)
    ap.add_argument("--dp", default="auto", choices=["auto", "p2p", "nccl"],
                    help="N > 1: fused reduce-scatter+Adam+all-gather over NVLink peer memory (p2p) or ncclAllReduce + "
                         "local Adam (nccl); auto = p2p when symmetric memory can be set up")
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / reference_gpu legs")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--no-balance", action="store_true", help="N > 1: plain round-robin view sharding instead of the "
                                                              "instance-count balanced one")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = --views-per-gpu views on every GPU; strong = the config's total view count "
                         "(8 for C3, 32 for C4) split over the GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (its loss and the parameters "
                         "after its Adam step, a fixed seeded sample of DUMP_ROWS Gaussians) as DIR/<name>.npy, float32")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this project's training step (--impl ours)")
    return a


DUMP_ROWS = 65536  # 59 floats per Gaussian at SH degree 3: ~15 MB per dump


def dump_last_step(tr, n: int, out_dir: str) -> None:
    """Writes the loss of the last step (summed over its views) and the parameters it left behind, for the rows of a fixed
    seeded sample of the Gaussians, so that two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch

    torch.cuda.synchronize()
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    idx = torch.as_tensor(rows, device=tr.device)
    out = {"loss": tr.loss_dev.detach().float().cpu().numpy()}
    for k, v in tr.export_params().items():
        out[k] = v.index_select(0, idx).float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(v, np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_leg(scene_obj, seconds: float):
    """The reference's path restated on the CPU (oracle port, OpenMP over all host cores) on a BOUNDED SAMPLE of the same
    workload: whole views (every Gaussian, every pixel of the 1920x1080 image; forward + L1/SSIM loss + backward) until
    `seconds` have passed -- at least one, at most three.  No crop and no extrapolation: value = views / time.  Adam is
    not included (it is < 1 % of a CPU view)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np

    import oracle as O

    sc = scene_obj
    cores = os.cpu_count() or 1
    W, H = sc.width, sc.height
    raw = dict(means=sc.means, sh0=sc.sh0, shN=sc.shN, scaling=sc.scaling, rotation=sc.rotation, opacity=sc.opacity)
    tgt = np.zeros((H, W, 3), np.uint8)
    t0 = time.time()
    reps = 0
    while True:
        v = reps % sc.viewmats.shape[0]
        O.view_loss_grads(raw, sc.viewmats[v], sc.Ks[v], W, H, sc.sh_degree, (0.0, 0.0, 0.0), target=tgt, prec=32,
                          lambda_dssim=LAMBDA_DSSIM)
        reps += 1
        if time.time() - t0 > seconds or reps >= 3:
            break
    dt = (time.time() - t0) / reps
    return {"value": 1.0 / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{reps} whole view(s): all {sc.n} Gaussians, all {W}x{H} pixels, fwd + L1/SSIM loss + bwd, "
                      f"{dt:.2f} s per view (no crop, no extrapolation; the Adam step is not in the sample)"}


def reference_gpu_leg(path: str, config: str, n_gaussians: int, views: int, steps: int, module: str = "ref"):
    """The reference's OWN training step on the same scene, cameras, loss and batch structure, in a child process:
    tools/ref_train.py drives oracle/ref_train_harness.cpp, i.e. the reference's FastGSRasterize (path 'fastgs') or
    SphericalHarmonicsFunction / fully_fused_projection_with_ut / GUTRasterizationFunction (path 'gut') autograd
    Functions, its fused_ssim and its FusedAdam, all compiled UNCHANGED, on the reference's own CUDA backends.  A
    baseline timed beside ours as the north_star asks -- never part of the product path.
    module 'b200': the SAME unchanged reference caller code linked against this library's host layer instead (the drop-in
    configuration a maintainer gets by switching the backend, INTEGRATION.md)."""
    cmd = [sys.executable, "-B", os.path.join(ROOT, "tools", "ref_train.py"), "--module", module, "--path", path,
           "--config", config, "--views", str(views), "--steps", str(max(2, min(steps, 4))), "--warmup", "2"]  # 2 warm-up steps: the
    # caching allocator needs them to hold a block for every per-view blob size (8 views, 4 blobs each)
    if n_gaussians:
        cmd += ["--n-gaussians", str(n_gaussians)]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    except subprocess.TimeoutExpired:
        return {"error": "timeout after 900 s"}
    got = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if got:
        d = json.loads(got[-1])
        if "value" not in d:
            d["error"] = ("the reference's forward_wrapper returned an implausible result on its first call "
                          "(profiles/r02_ref_fastgs_root_cause.txt)")
        return d
    tail = (r.stderr or r.stdout).strip().splitlines()
    return {"error": tail[-1][:300] if tail else f"exit code {r.returncode}"}


def stage_roofline(prof, n, I, P, deg, peak):
    """Algorithmic bytes per view of every stage (DESIGN.md section 4, BASELINE.md section 5 formulas) over its measured time,
    as a fraction of the measured HBM peak.  The blend stages are FP32/SFU-issue bound (their real DRAM traffic is a
    fraction of these bytes), the per-Gaussian and sort stages stream."""
    K = (deg + 1) ** 2
    G = float(n)
    bytes_of = {
        "preprocess_fwd": (44 + 12 * K + 12) * G + 96 * G,        # raw params + SH + GaussRec / CullRec / keys out
        "sort_intersect": 24 * G * 3 + 12 * I + 16 * I * 2 + 8 * I,  # 3 depth passes, emit, 2 tile passes, offsets
        "blend_fwd": 60 * I + 20 * P,
        "loss": 108 * P,
        "blend_bwd": 172 * I + 24 * P,
        "preprocess_bwd": (2 * 4 * (11 + 3 * K) + 64) * G,         # gradient planes read-modify-write + view accumulators
    }
    out = {}
    for k, b in bytes_of.items():
        ms = prof.get(k, 0.0)
        if ms > 0:
            gbs = b / (ms * 1e-3) / 1e9
            out[k] = {"algorithmic_bytes": b, "ms": ms, "GBps": gbs, "frac_of_hbm_peak": gbs / peak if peak else None}
    return out


# ------------------------------------------------------------------------------------------------------------------
def main():
    a = parse()
    import numpy as np
    from lichtfeld_studio_b200 import scene as S

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg_n, cfg_v, W, H, deg = S.CONFIGS[a.config]
    n = a.n_gaussians or cfg_n
    # C3 = 8 views per step on ONE GPU (BASELINE.json configs[2]); C4 = 32 views on 8 GPUs (configs[3]: 4 per GPU) with
    # eval/mcmc_optimization_params.json (opacity_reg = scale_reg = 0.01, src/training/trainer.cpp:132-158)
    base_vpg = {"C3": 8, "C4": 4}.get(a.config, cfg_v)
    if a.scaling == "strong":
        V = a.views_per_gpu * max(world, 1) if a.views_per_gpu else cfg_v
        V = max(V, world)
        vpg = (V + world - 1) // max(world, 1)
    else:
        vpg = a.views_per_gpu or base_vpg
        V = vpg * max(world, 1)
    mcmc = a.config == "C4"
    scale_reg = opacity_reg = 0.01 if mcmc else 0.0
    workload = (f"{a.config}: {n} Gaussians, {V} views per step ({a.scaling} scaling: {vpg} per GPU x {max(world, 1)} GPU) of "
                f"{W}x{H}, SH degree {deg}, 3DGUT from-world rasterizer, L1 + fused-SSIM loss (lambda_dssim {LAMBDA_DSSIM}), "
                + ("eval/mcmc_optimization_params.json (opacity_reg = scale_reg = 0.01 folded into the Adam step)" if mcmc
                   else "eval/default_optimization_params.json lrs"))

    if a.impl == "reference":
        # reference arm (tier rule): the reference's path on the box's host cores -- rank 0 only.  One "step" of this arm
        # is a bounded sample of the workload: ONE whole view (all Gaussians, all pixels) instead of the batch.
        if rank != 0:
            return 0
        sc = S.make_scene(n, 1, W, H, deg, seed=42)
        t_all = time.time()
        k = max(1, min(a.steps, 3))
        for _ in range(min(a.warmup, 1)):
            cpu_reference_leg(sc, 0.0)
        vals = [cpu_reference_leg(sc, 0.0) for _ in range(k)]
        cb = dict(vals[-1])
        cb["value"] = statistics.median(v["value"] for v in vals)
        cb["sample"] = f"{k} step(s) of ONE whole view each (all {n} Gaussians, all {W}x{H} pixels, fwd + L1/SSIM loss + bwd); " \
                       f"value = 1 view / median step time; no crop, no extrapolation"
        line = {"metric": METRIC, "value": cb["value"], "unit": UNIT, "impl": "reference", "n_gpus": a.gpus,
                "steps": k, "warmup": min(a.warmup, 1), "ms_per_step": 1e3 / cb["value"] if cb["value"] else None,
                "views_per_step": 1, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": workload + "; CPU port of the reference path (the reference has no CPU implementation "
                                                  "of the blend: tests/test_rasterization.cpp:96-98), one view per step",
                           "gaussians": n, "views_per_step": 1, "width": W, "height": H, "sh_degree": deg},
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "wall_s": round(time.time() - t_all, 1)}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from lichtfeld_studio_b200.trainer import SplatTrainer

    torch.cuda.set_device(local_rank)
    device = torch.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    sc = S.make_scene(n, V, W, H, deg, seed=42)
    my_views = list(range(rank, V, world))

    tr = SplatTrainer(n, W, H, deg, device, scale_reg=scale_reg, opacity_reg=opacity_reg)
    tr.load_scene(sc)
    tr.iteration = 1000  # steady state: the reference skips the shN group only for iteration <= 1000
    tr._dp_world = world
    # capacity calibration (one blocking forward per local view) -- outside every timed region
    tr.ensure_capacity([sc.viewmats[v] for v in my_views], [sc.Ks[v] for v in my_views], deg)
    n_inst_per_view = []
    for v in my_views:
        tr.forward(sc.viewmats[v], sc.Ks[v], deg)
        n_inst_per_view.append(tr.stats()[0])
    view_costs = None
    if world > 1 and not a.no_balance:
        # cost-balanced sharding: the tile-instance count of a camera (known from its last visit in a real run, from the
        # calibration pass here) predicts its render time; every rank gets the same number of views
        mine = torch.zeros(V, dtype=torch.float64, device=device)
        for v, c in zip(my_views, n_inst_per_view):
            mine[v] = float(c)
        dist.all_reduce(mine, op=dist.ReduceOp.SUM)
        view_costs = mine.cpu().tolist()
        from lichtfeld_studio_b200 import dp as _dp
        my_views = _dp.shard_views(V, world, rank, view_costs)
        tr.ensure_capacity([sc.viewmats[v] for v in my_views], [sc.Ks[v] for v in my_views], deg)
        n_inst_per_view = [view_costs[v] for v in my_views]

    dp_mode = "single"
    if world > 1:
        dp_mode = "nccl all-reduce of the flat gradient arena + local Adam"
        if a.dp in ("auto", "p2p"):
            try:
                tr.enable_p2p()
                dp_mode = ("fused reduce-scatter + Adam + all-gather in one kernel (lfs_adam_step_multi_p2p), " +
                           ("NVSwitch multicast: multimem.ld_reduce / multimem.st" if tr._mc_grads
                            else "NVLink peer loads / stores"))
            except Exception as e:  # symmetric memory unavailable on this box: the NCCL path is the validated fallback
                if a.dp == "p2p":
                    raise
                dp_mode += f" (p2p unavailable: {type(e).__name__})"
        flag = torch.tensor([1 if tr.p2p else 0], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)  # all ranks or none
        if int(flag.item()) == 0:
            tr.p2p = False
    targets_host = [torch.as_tensor(S.make_target(v, W, H)).pin_memory() for v in range(V)]
    targets_dev = {v: targets_host[v].to(device) for v in my_views}
    bg = (0.0, 0.0, 0.0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    targets_resident = [targets_dev.get(v, targets_host[v]) for v in range(V)]

    def step_resident():  # same public call as the e2e leg, targets already in HBM, loss left on the device
        tr.train_step(sc.viewmats, sc.Ks, targets_resident, bg, deg, world, rank, read_loss=False,
                      lambda_dssim=LAMBDA_DSSIM, view_costs=view_costs)

    def step_e2e():
        tr.train_step(sc.viewmats, sc.Ks, targets_host, bg, deg, world, rank, read_loss=True, view_costs=view_costs)
        torch.cuda.current_stream().synchronize()  # the step's result (loss) is read on the host

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = tr.lib.lfs_launch_count()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        launches = tr.lib.lfs_launch_count() - l0
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms.item()), int(launches)

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms_step, launches = timed(step_resident, a.steps, a.warmup)
    clk = clocks.stop() if rank == 0 else {}
    if a.dump_outputs and rank == 0:  # the later legs step the same parameters again
        dump_last_step(tr, n, a.dump_outputs)
    ms_e2e, _ = timed(step_e2e, a.steps, max(1, a.warmup))

    # per-kernel timing for the roofline: a PROFILING pass outside the timed regions.  Every stage is bracketed by CUDA
    # events and the backward blocks on the stream, so consecutive views do not overlap here: the stage times sum to a
    # little more than ms_per_step / views (in the timed run the tail of a view overlaps the head of the next).
    tr.lanes_enabled = False  # stage times: one view at a time (the timed runs keep tr.n_lanes views in flight)
    tr.set_profile(True)
    for _ in range(2):
        step_resident()
    torch.cuda.synchronize()
    prof = tr.get_profile()
    tr.set_profile(False)
    tr.lanes_enabled = True

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peak_gbs()
    I = float(np.mean(n_inst_per_view)) if n_inst_per_view else 0.0
    P = float(W * H)
    bwd_bytes = 172.0 * I + 24.0 * P
    fwd_bytes = 60.0 * I + 20.0 * P
    bwd_ms = prof.get("blend_bwd", 0.0)
    achieved = bwd_bytes / (bwd_ms * 1e-3) / 1e9 if bwd_ms > 0 else 0.0
    h2d = sum(int(targets_host[v].numel()) for v in my_views) + len(my_views) * (16 + 9) * 4
    # DRAM traffic of the same kernel from the committed `ncu --set full` capture of tools/profile_view.py on this
    # workload (ncu cannot run inside a timed bench): newest profiles/rNN_ncu_full*.json that has the kernel
    traffic, traffic_src = None, None
    import glob
    for path in (sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full*.json")), reverse=True)
                 if a.config == "C3" else []):  # the capture is of the C3 view
        try:
            for k in json.load(open(path)):
                if k["kernel"].startswith("k_blend_bwd"):
                    traffic = (k["dram__bytes_read.sum"] + k["dram__bytes_write.sum"]) * 1e6  # ncu reports Mbyte
                    traffic_src = f"profiles/{os.path.basename(path)} (dram__bytes_read.sum + dram__bytes_write.sum)"
                    break
        except (OSError, KeyError, ValueError, TypeError):
            continue
        if traffic is not None:
            break
    arena_bytes = int(tr.params.numel()) * 4
    line = {
        "metric": METRIC, "value": V / ms_step * 1e3, "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "gaussians": n, "views_per_step": V, "width": W, "height": H, "sh_degree": deg,
                   "parallelism": f"view-sharded dp{world}" + ("" if view_costs is None else " (views assigned by instance "
                                  "count, equal counts per rank)") + f": {dp_mode}",
                   "views_in_flight": tr.n_lanes, "instances_per_view": I, "l2": "per-step working set (params+grads+Adam state+records) >= 1 GB, "
                                                  "larger than the 126 MB L2: no flush needed"},
        "clocks": clk,
        "e2e": {"value": V / ms_e2e * 1e3, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4,
                "note": "SplatTrainer.train_step: pinned uint8 HWC targets copied per view on a side stream, "
                        "loss scalar read back per step"},
        "gpu_launches": launches,
        "roofline": {"kernel": "k_blend_bwd_sp", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src, "algorithmic_bytes": bwd_bytes, "launch_ms": bwd_ms,
                     "note": "algorithmic bytes = 172*I + 24*P per view (BASELINE.md s5); the kernel is FP32/SFU and "
                             "latency bound, not HBM bound (SURVEY s7 'roofline honesty')"},
        "stage_ms_per_view": prof,
        "stage_ms_note": "profiling pass with a blocking event pair per stage (views do not overlap): the sum exceeds "
                         "ms_per_step / views_per_gpu by the overlap the timed run gets",
        "stage_roofline": stage_roofline(prof, n, I, P, deg, peak),
    }
    if world > 1:
        # exchange step: every rank sends / receives (W-1)/W of the gradient arena (reduce-scatter) and of the parameter
        # arena (all-gather); the multicast variant receives 1/W of the gradients (reduced in the switch)
        line["nvlink"] = {"arena_bytes": arena_bytes,
                          "bytes_per_rank_per_step": 2.0 * (world - 1) / world * arena_bytes,
                          "note": "2 (W-1)/W x arena per rank per step (reduce-scatter + all-gather), the same volume an "
                                  "ncclAllReduce moves"}
    if not a.no_extras and world == 1:
        try:
            line["cpu_baseline"] = cpu_reference_leg(S.make_scene(n, 1, W, H, deg, seed=42), a.cpu_seconds)
        except Exception as e:
            line["cpu_baseline"] = {"error": repr(e)}
        try:  # separate processes: a fault inside a reference build must not take the bench down
            del tr
            torch.cuda.empty_cache()
            line["reference_gpu"] = {}
            for name, path in (("gsplat", "gut"), ("fastgs", "fastgs")):
                line["reference_gpu"][name] = reference_gpu_leg(path, a.config, a.n_gaussians, vpg, a.steps)
            for name, key in (("gsplat", "vs_reference_gsplat"), ("fastgs", "vs_reference_fastgs")):
                v = line["reference_gpu"][name].get("value")
                line[key] = (line["value"] / v) if v else None
        except Exception as e:
            line["reference_gpu"] = {"error": repr(e)}
        try:  # drop-in: the reference's unchanged autograd Functions / fused_ssim / FusedAdam on THIS library's backend
            line["drop_in"] = {}
            for name, path in (("gsplat", "gut"), ("fastgs", "fastgs")):
                d = reference_gpu_leg(path, a.config, a.n_gaussians, vpg, a.steps, module="b200")
                ref_v = (line.get("reference_gpu") or {}).get(name, {}).get("value")
                if d.get("value") and ref_v:
                    d["vs_reference_same_callers"] = d["value"] / ref_v
                line["drop_in"][name] = d
        except Exception as e:
            line["drop_in"] = {"error": repr(e)}
        try:  # the EWA (fastgs) surface of this library on the same workload, op level (forward + backward per view)
            r = subprocess.run([sys.executable, "-B", os.path.join(ROOT, "tools", "bench_fastgs.py"), a.config, "2",
                                "2"], capture_output=True, text=True, timeout=300)
            got = [l for l in r.stdout.splitlines() if l.startswith("{")]
            line["fastgs_surface"] = (json.loads(got[-1]) if got
                                      else {"error": (r.stderr or r.stdout).strip().splitlines()[-1][:300]})
        except Exception as e:
            line["fastgs_surface"] = {"error": repr(e)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
