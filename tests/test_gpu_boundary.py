"""-m gpu: the drop-in boundary EXECUTED (VERDICT r1 item 6).

oracle/ref_train_harness.cpp holds the reference's own callers compiled unchanged -- FastGSRasterize
(fast_rasterizer_autograd.cpp), SphericalHarmonicsFunction / fully_fused_projection_with_ut / GUTRasterizationFunction
(rasterizer_autograd.cpp), FusedAdam (fused_adam.cpp), fused_ssim (ssim.cu) -- and is linked twice:
    ref_fastgs_torch   on the reference's own fastgs + gsplat CUDA objects
    b200_fastgs_torch  on oracle/_ref/libgsplat_backend_b200.so (this project's host layer)
Every test runs the same call through both modules and compares: all 10 gsplat:: ops, forward_wrapper /
backward_wrapper, adam_step_wrapper go through the host layer on the GPU (so libgsplat_backend_b200.so shows up in the
driver's native_so_loaded), with the reference's callers above it bit-for-bit the same object code.
Metric as in test_gpu_baseline_configs.py (maxnorm + element-wise pass fraction)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import gpu_diag as D  # noqa: E402
import ref_libs as R  # noqa: E402
from lichtfeld_studio_b200 import scene  # noqa: E402
from test_gpu_baseline_configs import gate, gate_render, strict  # noqa: E402

T = D.T
LRS = [0.00016, 0.0025, 0.0025 / 20, 0.005, 0.001, 0.05]


@pytest.fixture(scope="module", autouse=True)
def _need_cuda_and_refs():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    R.require_all()


@pytest.fixture(scope="module")
def mods():
    return R.fastgs_torch_module("ref"), R.fastgs_torch_module("b200")


def _scene(n=20000, w=400, h=304, deg=3, views=2, seed=17):
    sc = scene.make_scene(n, views, w, h, deg, seed=seed, sigma_px=4.0)
    P = [T(sc.means), T(sc.sh0), T(sc.shN), T(sc.scaling), T(sc.rotation), T(sc.opacity.reshape(-1, 1))]
    cams = []
    for v in range(views):
        vm = sc.viewmats[v].astype(np.float64)
        cams.append(dict(w2c=T(sc.viewmats[v]), campos=T(-vm[:3, :3].T @ vm[:3, 3]), viewmat=T(sc.viewmats[v:v + 1]),
                         K=T(sc.Ks[v:v + 1]), k=[float(sc.Ks[v, 0, 0]), float(sc.Ks[v, 1, 1]), float(sc.Ks[v, 0, 2]),
                                                  float(sc.Ks[v, 1, 2])],
                         gt=T(scene.make_target(v, w, h)).permute(2, 0, 1).div(255.0).contiguous()))
    return sc, P, cams


GRADS = ("means", "sh0", "shN", "scaling", "rotation", "opacity")


def test_fastgs_callers_on_both_backends(mods):
    ref, b200 = mods
    sc, P, cams = _scene()
    bg = T(np.array([0.1, 0.2, 0.3]))
    rep = {}
    hr, hb = ref.Harness(*P, LRS), b200.Harness(*P, LRS)
    c = cams[0]
    nb = (sc.sh_degree + 1) ** 2
    a = hr.view_grads(c["w2c"], c["campos"], c["k"], c["gt"], bg, 0.2, nb, sc.width, sc.height)
    b = hb.view_grads(c["w2c"], c["campos"], c["k"], c["gt"], bg, 0.2, nb, sc.width, sc.height)
    # one (tile, primitive) instance on the boundary of the exact tile test, or one glitch of the reference's racy instance
    # creation (see test_gpu_baseline_configs._fastgs_vs_reference), moves up to 256 pixels and one primitive's gradients:
    # the element-wise fractions are the gate, the per-tensor maxima are bounded by one such event
    gate_render(rep, "image", b[0], a[0], min_frac=0.999)
    gate_render(rep, "alpha", b[1], a[1], min_frac=0.999)
    assert abs(float(a[2]) - float(b[2])) <= 1e-5 * abs(float(a[2])), (float(a[2]), float(b[2]))
    for name, x, y in zip(GRADS, b[3:], a[3:]):
        mn, fr = strict(x, y, 1e-3)
        rep["grad_" + name] = {"maxnorm": mn, "elementwise_pass_frac": fr, "rtol": 1e-3}
        assert fr >= 0.999 and mn <= 1e-2, (name, rep["grad_" + name])
    assert int((hr.densification_info[0] != hb.densification_info[0]).sum()) <= 2  # visibility counts
    gate(rep, "densification_norm", hb.densification_info[1], hr.densification_info[1], 1e-3, 0.99)
    print("fastgs callers:", rep)


def test_fastgs_training_steps_on_both_backends(mods):
    """Three optimiser steps (two views each, crossing iteration 1000 -> 1001 where FusedAdam starts stepping shN) of the
    reference's loop on both backends: the parameters must stay together."""
    ref, b200 = mods
    sc, P, cams = _scene()
    bg = T(np.zeros(3))
    hr, hb = ref.Harness(*P, LRS), b200.Harness(*P, LRS)
    nb = (sc.sh_degree + 1) ** 2
    args = ([c["w2c"] for c in cams], [c["campos"] for c in cams], [c["k"] for c in cams], [c["gt"] for c in cams], bg, 0.2,
            nb, sc.width, sc.height, True)
    for it in (999, 1000, 1001):
        lr_, lb_ = hr.train_step(it, *args), hb.train_step(it, *args)
        assert abs(lr_ - lb_) <= 1e-4 * abs(lr_), (it, lr_, lb_)
    rep = {}
    for name, x, y, p0 in zip(GRADS, hb.params(), hr.params(), P):
        # Adam's first steps move every parameter by ~lr * sign(g): compare the UPDATES
        # (an entry whose gradient is rounding noise around zero may step the other way: +-lr against -+lr, i.e. up to 2 x
        # the largest update; measured 0.008 % of the entries, largest deviation 2.7 % of the largest update)
        mn, fr = strict(x - p0, y - p0, 2e-2)
        rep["update_" + name] = {"maxnorm": mn, "elementwise_pass_frac": fr, "rtol": 2e-2}
        assert fr >= 0.999 and mn <= 2.0, (name, rep["update_" + name])
    print("fastgs training steps:", rep)


def test_gut_callers_on_both_backends(mods):
    ref, b200 = mods
    sc, P, cams = _scene(n=12000, w=320, h=240)
    bg = T(np.array([0.1, 0.2, 0.3]))
    rep = {}
    hr, hb = ref.GutHarness(*P, LRS), b200.GutHarness(*P, LRS)
    c = cams[0]
    a = hr.view_grads(c["viewmat"], c["K"], c["gt"], bg, 0.2, sc.sh_degree, sc.width, sc.height, 0)
    b = hb.view_grads(c["viewmat"], c["K"], c["gt"], bg, 0.2, sc.sh_degree, sc.width, sc.height, 0)
    assert hr.last_n_isects > 50_000 and abs(hr.last_n_isects - hb.last_n_isects) <= 2 + hr.last_n_isects // 2000
    # whole pipeline on each side's own projection: a radius that rounds the other way adds / removes a tile instance
    # (+-1 px is the reference's own tolerance), hence 5e-4 here; the per-stage gates on identical inputs are 1e-4
    gate_render(rep, "image", b[0], a[0], 5e-4)
    gate_render(rep, "alpha", b[1], a[1], 5e-4)
    assert abs(float(a[3]) - float(b[3])) <= 1e-4 * abs(float(a[3]))
    for name, x, y in zip(GRADS, b[4:], a[4:]):
        gate(rep, "grad_" + name, x, y, 2e-3, 0.98)
    print("3DGUT callers:", rep)


# (The reference's GUTRasterizationFunction refuses anything but three colour channels -- "Only 3 colors are supported
# currently", rasterizer_autograd.cpp -- so the RGB_D / D render modes of rasterize() cannot be exercised through its own
# autograd path; the op-level test below covers channels = 4 and 1 on both backends.)


def test_densification_ops_on_both_backends(mods):
    """relocation / add_noise / quats_to_rotmats (gsplat/RelocationCUDA.cu:12,113, QuatToRotmatCUDA.cu:14)."""
    ref, b200 = mods
    rng = np.random.RandomState(5)
    n, n_max = 50_000, 51
    q = T(rng.normal(size=(n, 4)))
    gate({}, "quats_to_rotmats", b200.quats_to_rotmats(q), ref.quats_to_rotmats(q), 1e-5, 0.999)
    op = T(rng.uniform(0.01, 0.99, size=n))
    sc = T(np.exp(rng.normal(-3, 1, size=(n, 3))))
    ratios = torch.as_tensor(rng.randint(1, n_max, size=n), dtype=torch.int32, device="cuda")
    import math
    binoms = np.zeros((n_max, n_max), np.float32)
    for i in range(n_max):
        for k in range(i + 1):
            binoms[i, k] = math.comb(i, k)
    bt = T(binoms)
    ro, rs = ref.relocation(op, sc, ratios, bt, n_max)
    bo, bs = b200.relocation(op, sc, ratios, bt, n_max)
    gate({}, "relocation_opacity", bo, ro, 1e-5, 0.999)
    gate({}, "relocation_scales", bs, rs, 1e-4, 0.999)
    raw_op, raw_sc, raw_q = T(rng.normal(size=n)), T(rng.normal(-3, 1, size=(n, 3))), T(rng.normal(size=(n, 4)))
    noise = T(rng.normal(size=(n, 3)))
    m_ref = T(rng.normal(size=(n, 3)))
    m_b = m_ref.clone()
    ref.add_noise(raw_op, raw_sc, raw_q, noise, m_ref, 1e-3)
    b200.add_noise(raw_op, raw_sc, raw_q, noise, m_b, 1e-3)
    gate({}, "add_noise_means", m_b, m_ref, 1e-6, 0.999)


def test_intersect_ops_on_both_backends(mods):
    ref, b200 = mods
    rng = np.random.RandomState(3)
    Cc, N, W, H = 2, 20000, 640, 480
    tw, th = (W + 15) // 16, (H + 15) // 16
    m2d = T((rng.uniform(-0.1, 1.1, size=(Cc, N, 2)) * np.array([W, H])))
    radii = torch.as_tensor(rng.randint(0, 30, size=(Cc, N, 2)), dtype=torch.int32, device="cuda")
    dep = T(rng.uniform(0.1, 20.0, size=(Cc, N)))
    a = ref.intersect_tile(m2d, radii, dep, Cc, 16, tw, th, True)
    b = b200.intersect_tile(m2d, radii, dep, Cc, 16, tw, th, True)
    for x, y in zip(a, b):
        assert x.shape == y.shape and torch.equal(x, y)
    assert torch.equal(ref.intersect_offset(a[1], Cc, tw, th), b200.intersect_offset(b[1], Cc, tw, th))
    # packed layout (gsplat/Intersect.cpp:32-39): a shuffled subset of the elements, each with its camera id
    sel = torch.as_tensor(rng.permutation(Cc * N)[: Cc * N // 2].copy(), device="cuda")
    pm, pr, pd = m2d.reshape(-1, 2)[sel].contiguous(), radii.reshape(-1, 2)[sel].contiguous(), dep.reshape(-1)[sel].contiguous()
    cam, gid = (sel // N).contiguous(), (sel % N).contiguous()
    for srt in (True, False):
        a = ref.intersect_tile_packed(pm, pr, pd, cam, gid, Cc, 16, tw, th, srt)
        b = b200.intersect_tile_packed(pm, pr, pd, cam, gid, Cc, 16, tw, th, srt)
        assert a[1].numel() > 10000
        for x, y in zip(a, b):
            assert x.shape == y.shape and torch.equal(x, y), srt


CAMERA_CASES = [
    dict(name="opencv_radial_tangential", model=0, rs=4, radial=[-0.12, 0.03, 0.002, 0.01, -0.004, 0.0005],
         tangential=[0.002, -0.0015], prism=None, vm1=False),
    dict(name="opencv_thin_prism", model=0, rs=4, radial=[-0.05, 0.01, 0.0, 0.0, 0.0, 0.0], tangential=None,
         prism=[0.003, -0.001, -0.002, 0.0005], vm1=False),
    dict(name="fisheye", model=2, rs=4, radial=[-0.02, 0.004, -0.0006, 0.00003], tangential=None, prism=None, vm1=False),
    dict(name="fisheye_k4_zero", model=2, rs=4, radial=[0.05, -0.01, 0.002, 0.0], tangential=None, prism=None, vm1=False),
    dict(name="pinhole_rolling_top_bottom", model=0, rs=0, radial=None, tangential=None, prism=None, vm1=True),
    dict(name="pinhole_rolling_right_left", model=0, rs=3, radial=None, tangential=None, prism=None, vm1=True),
    dict(name="fisheye_rolling_left_right", model=2, rs=1, radial=[-0.02, 0.004, 0.0, 0.0], tangential=None, prism=None,
         vm1=True),
    dict(name="opencv_rolling_bottom_top", model=0, rs=2, radial=[-0.08, 0.02, 0.0, 0.0, 0.0, 0.0],
         tangential=[0.001, 0.001], prism=None, vm1=True),
]


@pytest.mark.parametrize("case", CAMERA_CASES, ids=[c["name"] for c in CAMERA_CASES])
def test_projection_camera_models_on_both_backends(mods, case):
    """gsplat::projection_ut_3dgs_fused for the camera models the 3DGUT path exists for (gsplat/Cameras.cuh:416-1024:
    OpenCV pinhole distortion, fisheye) and rolling shutter (:346-413), host layer vs the reference CUDA build."""
    ref, b200 = mods
    n, w, h = 30000, 640, 480
    sc = scene.make_scene(n, 2, w, h, 0, seed=23, sigma_px=4.0)
    means, q, s, op, _ = sc.activated()
    vm0 = T(sc.viewmats[:1])
    vm1 = None
    if case["vm1"]:  # end-of-frame pose: a small rotation about y plus a translation
        a = 0.03
        d = np.array([[np.cos(a), 0, np.sin(a), 0.02], [0, 1, 0, -0.01], [-np.sin(a), 0, np.cos(a), 0.015], [0, 0, 0, 1]])
        vm1 = T((d @ sc.viewmats[0].astype(np.float64))[None])
    K = sc.Ks[:1].copy()
    if case["model"] == 2:
        K[0, 0, 0] = K[0, 1, 1] = 0.45 * w  # wide field of view
    opt = lambda v: None if v is None else T(np.array([v], np.float32))  # noqa: E731
    args = (T(means), T(q), T(s), T(op), vm0, vm1, T(K), w, h, 0.3, 0.01, 1e4, 0.0, True, case["model"], case["rs"],
            opt(case["radial"]), opt(case["tangential"]), opt(case["prism"]))
    a_ = ref.projection_ut(*args)
    b_ = b200.projection_ut(*args)
    rr, rb = a_[0], b_[0]
    vis_r, vis_b = (rr > 0).all(-1), (rb > 0).all(-1)
    n_vis = int(vis_r.sum())
    assert n_vis > 2000, (case["name"], n_vis)
    both = vis_r & vis_b
    rolling = case["rs"] != 4
    # Rolling shutter: every sigma point is projected through its own pose, glm::slerp(q_start, q_end, t) with
    # t = floor(pixel row or column) / (size - 1) re-evaluated in 10 fixed-point iterations (Cameras.cuh:293-318, :391-407).
    # The reference evaluates the slerp with --use_fast_math, i.e. sin.approx, whose absolute error is ~2e-5 RELATIVE for the
    # small angle between the two poses; the seven points get independent errors, and the UT weights (-99, 7 x 16.7) turn
    # them into pixels.  The exact-sinf projection differs from the reference by the reference's noise alone (measured:
    # >= 98 % of the means inside 1e-4, radii off by up to 5 px on 0.8 % of the Gaussians); reproducing sin.approx here makes
    # it worse (61 %), the noise only cancels for bit-identical code.  Depth is taken at the mid-frame pose -- one slerp with
    # the same inputs for every Gaussian -- and is reproduced with the reference's arithmetic (projection.cuh).
    vis_tol, frac, rdiff = (n_vis // 100, 0.97, 6) if rolling else (max(3, n_vis // 500), 0.999, 1)
    rep = {"n_visible": n_vis, "visibility_mismatch": int((vis_r != vis_b).sum()),
           "radii_max_diff": int((rr[both] - rb[both]).abs().max()),
           "radii_diff_gt1_frac": float(((rr[both] - rb[both]).abs() > 1).any(-1).float().mean())}
    assert rep["visibility_mismatch"] <= vis_tol and rep["radii_max_diff"] <= rdiff, (case["name"], rep)
    assert rep["radii_diff_gt1_frac"] <= (1e-2 if rolling else 0.0), (case["name"], rep)
    for key, idx, rtol in (("means2d", 1, 1e-4), ("depths", 2, 1e-5), ("conics", 3, 2e-3), ("compensations", 4, 1e-3)):
        mn, fr = strict(b_[idx][both], a_[idx][both], rtol)
        rep[key] = {"maxnorm": mn, "elementwise_pass_frac": fr, "rtol": rtol}
        # conics / compensations: second moments of the same noisy points (measured 93-95 % inside 2e-3 with rolling shutter)
        assert fr >= (frac if key in ("means2d", "depths") else (0.90 if rolling else 0.98)), (case["name"], key, rep[key])
        if not rolling:
            assert mn <= rtol, (case["name"], key, rep[key])
    print(case["name"], n_vis, rep)


@pytest.mark.parametrize("case", CAMERA_CASES, ids=[c["name"] for c in CAMERA_CASES])
def test_rasterize_camera_models_on_both_backends(mods, case):
    """rasterize_to_pixels_from_world_3dgs_fwd / _bwd along per-pixel rays (distortion, fisheye, rolling shutter): host
    layer vs the reference CUDA build, both on the reference's own projection + tile lists."""
    ref, b200 = mods
    n, w, h = 12000, 320, 240
    sc = scene.make_scene(n, 2, w, h, 0, seed=29, sigma_px=4.0)
    means, q, s, op, _ = sc.activated()
    vm0 = T(sc.viewmats[:1])
    vm1 = None
    if case["vm1"]:
        a = 0.03
        d = np.array([[np.cos(a), 0, np.sin(a), 0.02], [0, 1, 0, -0.01], [-np.sin(a), 0, np.cos(a), 0.015], [0, 0, 0, 1]])
        vm1 = T((d @ sc.viewmats[0].astype(np.float64))[None])
    K = sc.Ks[:1].copy()
    if case["model"] == 2:
        K[0, 0, 0] = K[0, 1, 1] = 0.45 * w
    opt = lambda v: None if v is None else T(np.array([v], np.float32))  # noqa: E731
    rad, tan, pri = opt(case["radial"]), opt(case["tangential"]), opt(case["prism"])
    tm, tq, ts, to, tK = T(means), T(q), T(s), T(op), T(K)
    radii, m2d, dep, con, _ = ref.projection_ut(tm, tq, ts, to, vm0, vm1, tK, w, h, 0.3, 0.01, 1e4, 0.0, False,
                                                case["model"], case["rs"], rad, tan, pri)
    tw, th = (w + 15) // 16, (h + 15) // 16
    _, ids, flat = ref.intersect_tile(m2d, radii, dep, 1, 16, tw, th, True)
    offs = ref.intersect_offset(ids, 1, tw, th)
    assert flat.numel() > 20_000
    g = torch.Generator(device="cuda").manual_seed(4)
    colors = torch.rand((1, n, 3), device="cuda", generator=g)
    bg = T(np.array([[0.1, 0.2, 0.3]]))
    fargs = (tm, tq, ts, colors, to[None].contiguous(), bg, w, h, vm0, vm1, tK, case["model"], case["rs"], rad, tan, pri,
             offs, flat)
    a_ = ref.raster_fwd(*fargs)
    b_ = b200.raster_fwd(*fargs)
    rep = {}
    # Rolling shutter: every pixel has its own pose, glm::slerp of the two frame poses evaluated with the reference's
    # --use_fast_math sin.approx (cameras.cuh quat_slerp<true> reproduces it; with exact sinf only 83 % of the render is inside
    # the 1e-4 band).  What is left is the last bit of the sin.approx ARGUMENTS (FMA contraction, div.approx of the frame
    # time), which moves single rays by ~1e-4 of a Gaussian's extent: measured 99.7 % inside the band, worst value 2e-3.
    rolling = case["rs"] != 4
    gate_render(rep, "render_rgb", b_[0], a_[0], min_frac=0.995 if rolling else 0.9999)
    gate_render(rep, "render_alpha", b_[1], a_[1], min_frac=0.995 if rolling else 0.9999)
    assert float((a_[2] != b_[2]).float().mean()) <= 2e-3
    vC = torch.randn(a_[0].shape, device="cuda", generator=g)
    vA = torch.randn(a_[1].shape, device="cuda", generator=g)
    ga = ref.raster_bwd(*fargs, a_[1], a_[2], vC, vA)
    gb = b200.raster_bwd(*fargs, b_[1], b_[2], vC, vA)
    for nm, x, y in zip(("v_means", "v_quats", "v_scales", "v_colors", "v_opacities"), gb, ga):
        gate(rep, "bwd_" + nm, x, y, 5e-3 if rolling else 1e-3, 0.99)  # rolling: measured 3.3e-3 on v_quats (see above)
    print(case["name"], int(flat.numel()), rep)


def test_rasterize_four_channels_on_both_backends(mods):
    """channels = 4 (RGB + depth, rasterizer.cpp:272-300) and 1 (depth only) through the op surface."""
    ref, b200 = mods
    n, w, h = 8000, 256, 192
    sc = scene.make_scene(n, 1, w, h, 0, seed=31, sigma_px=4.0)
    means, q, s, op, _ = sc.activated()
    tm, tq, ts, to, tK, vm0 = T(means), T(q), T(s), T(op), T(sc.Ks[:1]), T(sc.viewmats[:1])
    radii, m2d, dep, con, _ = ref.projection_ut(tm, tq, ts, to, vm0, None, tK, w, h, 0.3, 0.01, 1e4, 0.0, False, 0, 4, None,
                                                None, None)
    tw, th = (w + 15) // 16, (h + 15) // 16
    _, ids, flat = ref.intersect_tile(m2d, radii, dep, 1, 16, tw, th, True)
    offs = ref.intersect_offset(ids, 1, tw, th)
    g = torch.Generator(device="cuda").manual_seed(5)
    for ch in (4, 1):
        colors = torch.rand((1, n, ch), device="cuda", generator=g)
        bg = torch.rand((1, ch), device="cuda", generator=g)
        fargs = (tm, tq, ts, colors, to[None].contiguous(), bg, w, h, vm0, None, tK, 0, 4, None, None, None, offs, flat)
        a_, b_ = ref.raster_fwd(*fargs), b200.raster_fwd(*fargs)
        rep = {}
        gate_render(rep, "render", b_[0], a_[0])
        gate_render(rep, "alpha", b_[1], a_[1])
        vC = torch.randn(a_[0].shape, device="cuda", generator=g)
        vA = torch.randn(a_[1].shape, device="cuda", generator=g)
        ga = ref.raster_bwd(*fargs, a_[1], a_[2], vC, vA)
        gb = b200.raster_bwd(*fargs, b_[1], b_[2], vC, vA)
        for nm, x, y in zip(("v_means", "v_quats", "v_scales", "v_colors", "v_opacities"), gb, ga):
            gate(rep, f"bwd_{nm}", x, y, 1e-3, 0.99)
        print("channels", ch, rep)
