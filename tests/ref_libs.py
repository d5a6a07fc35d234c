"""ctypes front-ends of the UNMODIFIED reference builds under oracle/_ref/ (TEST INFRASTRUCTURE ONLY).

  libgsplat_ref.so  -- /root/reference/gsplat/*.cu,*.cpp compiled against oracle/glm_shim   (GPU)
  libfastgs_ref.so  -- /root/reference/fastgs/**                                            (GPU)
Built in the build container by `make -C oracle ref`; they travel to the GPU box with the snapshot.
All functions take / return torch CUDA tensors.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_REF = os.path.join(_ROOT, "oracle", "_ref")
_gs = None
_fg = None


def have_gsplat() -> bool:
    return os.path.exists(os.path.join(_REF, "libgsplat_ref.so"))


def have_fastgs() -> bool:
    return os.path.exists(os.path.join(_REF, "libfastgs_ref.so"))


def gsplat():
    global _gs
    if _gs is None:
        _gs = C.CDLL(os.path.join(_REF, "libgsplat_ref.so"))
        _gs.ref_gsplat_intersect_tile.restype = C.c_longlong
    return _gs


def fastgs():
    global _fg
    if _fg is None:
        _fg = C.CDLL(os.path.join(_REF, "libfastgs_ref.so"))
        _fg.ref_fastgs_create.restype = C.c_void_p
    return _fg


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _f32(t):
    return t.contiguous().float()


# ---------------------------------------------------------------------------------------------- gsplat reference
def projection_ut(means, quats, scales, opacities, viewmats, Ks, W, H, eps2d=0.3, near=0.01, far=1e4, clip=0.0,
                  calc_comp=False):
    N, Cc, dev = means.shape[0], Ks.shape[0], means.device
    radii = torch.zeros((Cc, N, 2), dtype=torch.int32, device=dev)
    m2d = torch.zeros((Cc, N, 2), device=dev)
    dep = torch.zeros((Cc, N), device=dev)
    con = torch.zeros((Cc, N, 3), device=dev)
    comp = torch.zeros((Cc, N), device=dev)
    rc = gsplat().ref_gsplat_projection_ut(_p(means), _p(quats), _p(scales), _p(opacities), _p(viewmats), _p(Ks),
                                           C.c_int(N), C.c_int(Cc), C.c_int(W), C.c_int(H), C.c_float(eps2d),
                                           C.c_float(near), C.c_float(far), C.c_float(clip), C.c_int(int(calc_comp)),
                                           _p(radii), _p(m2d), _p(dep), _p(con), _p(comp))
    assert rc == 0
    return radii, m2d, dep, con, comp


def sh_fwd(degree, dirs, coeffs, masks=None):
    n, K = dirs.shape[0], coeffs.shape[1]
    colors = torch.zeros((n, 3), device=dirs.device)
    rc = gsplat().ref_gsplat_sh_fwd(C.c_int(degree), _p(dirs), _p(coeffs), _p(masks), C.c_int(n), C.c_int(K),
                                    _p(colors))
    assert rc == 0
    return colors


def sh_bwd(degree, dirs, coeffs, v_colors, masks=None, compute_v_dirs=True):
    n, K = dirs.shape[0], coeffs.shape[1]
    v_coeffs = torch.zeros_like(coeffs)
    v_dirs = torch.zeros_like(dirs)
    rc = gsplat().ref_gsplat_sh_bwd(C.c_int(degree), _p(dirs), _p(coeffs), _p(masks), _p(v_colors), C.c_int(n),
                                    C.c_int(K), C.c_int(int(compute_v_dirs)), _p(v_coeffs), _p(v_dirs))
    assert rc == 0
    return v_coeffs, v_dirs


def intersect_tile(means2d, radii, depths, tile_size, tw, th, sort=True):
    Cc, N = depths.shape
    dev = depths.device
    tpg = torch.zeros((Cc, N), dtype=torch.int32, device=dev)
    cap = int(Cc * N * min(tw * th, 4096)) + 16
    ids = torch.zeros(cap, dtype=torch.int64, device=dev)
    flat = torch.zeros(cap, dtype=torch.int32, device=dev)
    n = gsplat().ref_gsplat_intersect_tile(_p(means2d), _p(radii), _p(depths), C.c_int(Cc), C.c_int(N),
                                           C.c_int(tile_size), C.c_int(tw), C.c_int(th), C.c_int(int(sort)), _p(tpg),
                                           _p(ids), _p(flat), C.c_longlong(cap))
    assert 0 <= n <= cap, n
    return tpg, ids[:n].clone(), flat[:n].clone()


def intersect_offset(isect_ids, Cc, tw, th):
    off = torch.zeros((Cc, th, tw), dtype=torch.int32, device=isect_ids.device)
    rc = gsplat().ref_gsplat_intersect_offset(_p(isect_ids), C.c_longlong(isect_ids.numel()), C.c_int(Cc), C.c_int(tw),
                                              C.c_int(th), _p(off))
    assert rc == 0
    return off


def raster_fwd(means, quats, scales, colors, opacities, backgrounds, W, H, tile_size, viewmats, Ks, tile_offsets,
               flatten_ids):
    Cc, N, dev = viewmats.shape[0], means.shape[0], means.device
    ren = torch.zeros((Cc, H, W, 3), device=dev)
    al = torch.zeros((Cc, H, W, 1), device=dev)
    li = torch.zeros((Cc, H, W), dtype=torch.int32, device=dev)
    rc = gsplat().ref_gsplat_raster_fwd(_p(means), _p(quats), _p(scales), _p(colors), _p(opacities), _p(backgrounds),
                                        C.c_int(N), C.c_int(Cc), C.c_int(3), C.c_int(W), C.c_int(H), C.c_int(tile_size),
                                        _p(viewmats), _p(Ks), _p(tile_offsets), _p(flatten_ids),
                                        C.c_longlong(flatten_ids.numel()), _p(ren), _p(al), _p(li))
    assert rc == 0
    return ren, al, li


def raster_bwd(means, quats, scales, colors, opacities, backgrounds, W, H, tile_size, viewmats, Ks, tile_offsets,
               flatten_ids, render_alphas, last_ids, v_colors_in, v_alphas_in):
    Cc, N, dev = viewmats.shape[0], means.shape[0], means.device
    vm = torch.zeros((N, 3), device=dev)
    vq = torch.zeros((N, 4), device=dev)
    vs = torch.zeros((N, 3), device=dev)
    vc = torch.zeros((Cc, N, 3), device=dev)
    vo = torch.zeros((Cc, N), device=dev)
    rc = gsplat().ref_gsplat_raster_bwd(_p(means), _p(quats), _p(scales), _p(colors), _p(opacities), _p(backgrounds),
                                        C.c_int(N), C.c_int(Cc), C.c_int(W), C.c_int(H), C.c_int(tile_size),
                                        _p(viewmats), _p(Ks), _p(tile_offsets), _p(flatten_ids),
                                        C.c_longlong(flatten_ids.numel()), _p(render_alphas), _p(last_ids),
                                        _p(v_colors_in), _p(v_alphas_in), _p(vm), _p(vq), _p(vs), _p(vc), _p(vo))
    assert rc == 0
    return vm, vq, vs, vc, vo


# ---------------------------------------------------------------------------------------------- fastgs reference
class FastGS:
    """fast_gs::rasterization::forward / backward + optimizer::adam_step through oracle/ref_fastgs_capi.cu."""

    def __init__(self):
        self.lib = fastgs()
        self.h = C.c_void_p(self.lib.ref_fastgs_create())

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_fastgs_destroy(self.h)
            self.h = None

    def forward(self, means, scales_raw, rot_raw, op_raw, sh0, shN, w2c, cam_pos, active_sh_bases, W, H, fx, fy, cx, cy,
                near=0.01, far=1e10):
        dev = means.device
        N = means.shape[0]
        image = torch.zeros((3, H, W), device=dev)
        alpha = torch.zeros((1, H, W), device=dev)
        counts = (C.c_int * 3)()
        rc = self.lib.ref_fastgs_forward(self.h, _p(means), _p(scales_raw), _p(rot_raw), _p(op_raw), _p(sh0), _p(shN),
                                         _p(w2c), _p(cam_pos), _p(image), _p(alpha), C.c_int(N),
                                         C.c_int(active_sh_bases), C.c_int(shN.shape[1]), C.c_int(W), C.c_int(H),
                                         C.c_float(fx), C.c_float(fy), C.c_float(cx), C.c_float(cy), C.c_float(near),
                                         C.c_float(far), counts)
        assert rc == 0, rc
        return image, alpha, tuple(counts)

    def backward(self, grad_image, grad_alpha, image, alpha, means, scales_raw, rot_raw, shN, w2c, cam_pos,
                 active_sh_bases, W, H, fx, fy, cx, cy, grads=None):
        dev = means.device
        N = means.shape[0]
        if grads is None:
            grads = dict(means=torch.zeros((N, 3), device=dev), scales=torch.zeros((N, 3), device=dev),
                         rot=torch.zeros((N, 4), device=dev), op=torch.zeros((N, 1), device=dev),
                         sh0=torch.zeros((N, 1, 3), device=dev), shN=torch.zeros_like(shN),
                         m2d=torch.zeros((N, 2), device=dev), conic=torch.zeros((3, N), device=dev))
        rc = self.lib.ref_fastgs_backward(self.h, _p(grad_image), _p(grad_alpha), _p(image), _p(alpha), _p(means),
                                          _p(scales_raw), _p(rot_raw), _p(shN), _p(w2c), _p(cam_pos),
                                          _p(grads["means"]), _p(grads["scales"]), _p(grads["rot"]), _p(grads["op"]),
                                          _p(grads["sh0"]), _p(grads["shN"]), _p(grads["m2d"]), _p(grads["conic"]),
                                          None, C.c_int(N), C.c_int(active_sh_bases), C.c_int(shN.shape[1]), C.c_int(W),
                                          C.c_int(H), C.c_float(fx), C.c_float(fy), C.c_float(cx), C.c_float(cy))
        assert rc == 0, rc
        return grads

    def adam_step(self, p, m, v, g, lr, b1, b2, eps, bc1, bc2):
        rc = self.lib.ref_fastgs_adam_step(_p(p), _p(m), _p(v), _p(g), C.c_int(p.numel()), C.c_float(lr), C.c_float(b1),
                                           C.c_float(b2), C.c_float(eps), C.c_float(bc1), C.c_float(bc2))
        assert rc == 0, rc


# ---------------------------------------------------------------------------------------------- presence gate
def require_all():
    """On a box with a CUDA device the reference builds MUST be present: a missing oracle/_ref/*.so would silently turn
    every 'vs the unmodified reference' assertion into a no-op (VERDICT r1, weak #3)."""
    import glob
    missing = [n for n in ("libgsplat_ref.so", "libfastgs_ref.so", "libtorch_impl_ref.so", "libgsplat_backend_b200.so")
               if not os.path.exists(os.path.join(_REF, n))]
    for mod in ("ref_fastgs_torch", "b200_fastgs_torch"):
        if not glob.glob(os.path.join(_REF, mod + "*.so")):
            missing.append(mod + "*.so")
    assert not missing, (f"reference builds missing under oracle/_ref: {missing} -- run `make -C oracle ref` in the build "
                         "container (they travel to the GPU box with the snapshot)")


_ti = None


def torch_impl():
    """UNMODIFIED /root/reference/tests/torch_impl.cpp (CPU ATen) behind oracle/ref_torch_impl_capi.cpp."""
    global _ti
    if _ti is None:
        _ti = C.CDLL(os.path.join(_REF, "libtorch_impl_ref.so"))
        _ti.ref_ti_isect_tiles.restype = C.c_longlong
    return _ti


def ti_spherical_harmonics(degree, dirs, coeffs):
    import numpy as np
    n, K = dirs.shape[0], coeffs.shape[1]
    out = np.zeros((n, 3), np.float32)
    d, c = np.ascontiguousarray(dirs, np.float32), np.ascontiguousarray(coeffs, np.float32)
    torch_impl().ref_ti_spherical_harmonics(C.c_int(degree), d.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p),
                                            C.c_int(n), C.c_int(K), out.ctypes.data_as(C.c_void_p))
    return out


def ti_isect_tiles(means2d, radii, depths, tile, tw, th, sort=True):
    import numpy as np
    Cc, N = depths.shape
    m, r, d = (np.ascontiguousarray(means2d, np.float32), np.ascontiguousarray(radii, np.int32),
               np.ascontiguousarray(depths, np.float32))
    # exact upper bound of the instance count: the AABB tile box of every Gaussian
    cap = int(Cc * N * 64) + 1024
    tpg = np.zeros((Cc, N), np.int32)
    ids = np.zeros(cap, np.int64)
    flat = np.zeros(cap, np.int32)
    k = torch_impl().ref_ti_isect_tiles(m.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p),
                                        d.ctypes.data_as(C.c_void_p), C.c_int(Cc), C.c_int(N), C.c_int(tile), C.c_int(tw),
                                        C.c_int(th), C.c_int(int(sort)), tpg.ctypes.data_as(C.c_void_p),
                                        ids.ctypes.data_as(C.c_void_p), flat.ctypes.data_as(C.c_void_p),
                                        C.c_longlong(cap))
    assert k <= cap, (k, cap)
    return tpg, ids[:k], flat[:k]


def fastgs_torch_module(which="ref"):
    """oracle/ref_train_harness.cpp built against the reference's fastgs objects ('ref') or against this project's host
    layer ('b200')."""
    import glob
    import importlib.util
    import sys
    name = {"ref": "ref_fastgs_torch", "b200": "b200_fastgs_torch"}[which]
    if name in sys.modules:  # a pybind11 module registers its types once per process
        return sys.modules[name]
    hits = glob.glob(os.path.join(_REF, name + "*.so"))
    assert hits, f"oracle/_ref/{name}*.so missing"
    if which == "b200":
        # the host layer the module links against, loaded by path so that the module resolves it by its soname whatever
        # run path the module was linked with
        C.CDLL(os.path.join(_REF, "libgsplat_backend_b200.so"), mode=C.RTLD_GLOBAL)
    spec = importlib.util.spec_from_file_location(name, hits[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.modules[name] = mod
    return mod
