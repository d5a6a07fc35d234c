"""Runs the reference's OWN training step (oracle/ref_train_harness.cpp: the FastGSRasterize / GUTRasterizationFunction /
SphericalHarmonicsFunction autograd Functions, fused_ssim, FusedAdam -- all compiled unchanged from /root/reference) on a
seeded BASELINE config, through

    --module ref    oracle/_ref/ref_fastgs_torch*.so   the reference's own CUDA backends          (the denominator)
    --module b200   oracle/_ref/b200_fastgs_torch*.so  this project's host layer as the backend   (boundary executed)
    --path fastgs   the default EWA rasterizer (fast_rasterize)      --path gut   the 3DGUT rasterizer (--gut)

    python tools/ref_train.py --module ref --path fastgs --config C3 --views 8 --steps 3 --warmup 1 [--check]

Prints one JSON line: views/s (CUDA events on the current stream, steps bracketed by synchronize), counts and a
plausibility check of the first forward (finite image, n_buckets consistent).  TEST / BENCH INFRASTRUCTURE ONLY."""
import argparse
import glob
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import ref_libs  # noqa: E402
from lichtfeld_studio_b200 import scene as S  # noqa: E402

LRS = [0.00016, 0.0025, 0.0025 / 20, 0.005, 0.001, 0.05]  # eval/default_optimization_params.json, FusedAdam group order


def load_module(which: str):
    name = {"ref": "ref_fastgs_torch", "b200": "b200_fastgs_torch"}[which]
    if not glob.glob(os.path.join(ROOT, "oracle", "_ref", name + "*.so")):
        raise FileNotFoundError(f"oracle/_ref/{name}*.so not built (make -C oracle fastgs_torchmod)")
    return ref_libs.fastgs_torch_module(which)


def scene_tensors(sc, dev):
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).to(dev)  # noqa: E731
    cams = []
    for v in range(sc.viewmats.shape[0]):
        vm = sc.viewmats[v].astype(np.float64)
        cams.append((T(sc.viewmats[v]), T(-vm[:3, :3].T @ vm[:3, 3]),
                     [float(sc.Ks[v, 0, 0]), float(sc.Ks[v, 1, 1]), float(sc.Ks[v, 0, 2]), float(sc.Ks[v, 1, 2])]))
    P = [T(sc.means), T(sc.sh0), T(sc.shN), T(sc.scaling), T(sc.rotation), T(sc.opacity.reshape(-1, 1))]
    return P, cams


def run_gut(a, mod, sc, P, out, dev, V, W, H, deg):
    """the reference's 3DGUT step: GutHarness = rasterize() of rasterizer.cpp on its own autograd Functions"""
    T = lambda x: torch.as_tensor(np.ascontiguousarray(x, np.float32)).to(dev)  # noqa: E731
    h = mod.GutHarness(*P, LRS)
    gts = [torch.as_tensor(S.make_target(v, W, H)).to(dev).permute(2, 0, 1).float().div_(255.0).contiguous()
           for v in range(V)]
    vms = [T(sc.viewmats[v:v + 1]) for v in range(V)]
    Ks = [T(sc.Ks[v:v + 1]) for v in range(V)]
    bg = torch.zeros(3, device=dev)
    it = 1001
    for i in range(a.warmup):
        h.train_step(it + i, vms, Ks, gts, bg, a.lambda_dssim, deg, W, H, False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss = 0.0
    for i in range(a.steps):
        loss = h.train_step(it + a.warmup + i, vms, Ks, gts, bg, a.lambda_dssim, deg, W, H, i == a.steps - 1)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    out.update({"value": V / ms * 1e3, "unit": "views/s", "ms_per_step": ms, "steps": a.steps, "warmup": a.warmup,
                "loss_last_step": loss, "instances_last_view": int(h.last_n_isects),
                "impl": ("reference gsplat (3DGUT) CUDA kernels + the reference's rasterizer_autograd.cpp / fused_ssim / "
                         "FusedAdam, all unmodified (kernels built against oracle/glm_shim)" if a.module == "ref" else
                         "the reference's rasterizer_autograd.cpp / fused_ssim / FusedAdam (unmodified) on this project's "
                         "host layer"),
                "note": "targets resident in HBM; L1 + fused SSIM loss; one FusedAdam::step per step"})
    print(json.dumps(out))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--module", default="ref", choices=["ref", "b200"])
    ap.add_argument("--path", default="fastgs", choices=["fastgs", "gut"])
    ap.add_argument("--config", default="C3")
    ap.add_argument("--n-gaussians", type=int, default=0)
    ap.add_argument("--views", type=int, default=0)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--lambda-dssim", type=float, default=0.2)
    ap.add_argument("--check", action="store_true", help="only the first-forward plausibility check")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    n, V, W, H, deg = S.CONFIGS[a.config]
    n = a.n_gaussians or n
    V = a.views or V
    sc = S.make_scene(n, V, W, H, deg, seed=42)
    mod = load_module(a.module)
    P, cams = scene_tensors(sc, dev)
    nb = (deg + 1) ** 2
    out = {"module": a.module, "path": a.path, "config": a.config, "gaussians": n, "views_per_step": V, "width": W,
           "height": H, "cudart": torch.version.cuda}
    if a.path == "gut":
        return run_gut(a, mod, sc, P, out, dev, V, W, H, deg)

    # 1. the reference's forward_wrapper, called directly, torch-owned blobs, nothing zero-filled, nothing swallowed
    w2c, cp, k = cams[0]
    r = mod.forward_wrapper(P[0], P[3], P[4], P[5], P[1], P[2], w2c, cp, nb, W, H, k[0], k[1], k[2], k[3], 0.01, 1e10)
    torch.cuda.synchronize()
    image, alpha, n_vis, n_inst, n_buckets = r[0], r[1], r[6], r[7], r[8]
    out["first_forward"] = {"n_visible": int(n_vis), "n_instances": int(n_inst), "n_buckets": int(n_buckets),
                            "image_finite": bool(torch.isfinite(image).all()), "image_mean": float(image.mean()),
                            "alpha_mean": float(alpha.mean()),
                            "plausible": bool(0 < n_buckets < n_inst // 8 + ((W + 15) // 16) * ((H + 15) // 16) + 1
                                              and torch.isfinite(image).all())}
    if a.check or not out["first_forward"]["plausible"]:
        print(json.dumps(out))
        return 0 if out["first_forward"]["plausible"] else 1
    del r, image, alpha

    # 2. the training step of the reference's callers
    h = mod.Harness(*P, LRS)
    gts = [torch.as_tensor(S.make_target(v, W, H)).to(dev).permute(2, 0, 1).float().div_(255.0).contiguous()
           for v in range(V)]
    bg = torch.zeros(3, device=dev)
    w2cs, cps, ks = [c[0] for c in cams], [c[1] for c in cams], [c[2] for c in cams]
    it = 1001  # steady state: FusedAdam skips the shN group only for iteration <= 1000 (fused_adam.cpp:69)
    for i in range(a.warmup):
        h.train_step(it + i, w2cs, cps, ks, gts, bg, a.lambda_dssim, nb, W, H, False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss = 0.0
    for i in range(a.steps):
        loss = h.train_step(it + a.warmup + i, w2cs, cps, ks, gts, bg, a.lambda_dssim, nb, W, H, i == a.steps - 1)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    out.update({"value": V / ms * 1e3, "unit": "views/s", "ms_per_step": ms, "steps": a.steps, "warmup": a.warmup,
                "loss_last_step": loss,
                "impl": ("reference fastgs (EWA) CUDA build + the reference's FastGSRasterize / fused_ssim / FusedAdam, "
                         "all unmodified" if a.module == "ref" else
                         "the reference's FastGSRasterize / fused_ssim / FusedAdam (unmodified) on this project's host layer"),
                "note": "targets resident in HBM; L1 + fused SSIM loss (lambda_dssim 0.2); gradients of the views of a "
                        "step accumulate in .grad, one FusedAdam::step per step"})
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
