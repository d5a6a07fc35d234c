"""The C++/libtorch host layer (lichtfeld-studio_b200/host/gsplat_backend.cpp, fastgs_adam_backend.cpp, fastgs_raster_backend.cpp) compiled
against the REFERENCE's own headers must export exactly the mangled symbols that the reference's own objects define
for its public operator surface (tests/golden/ref_symbols.txt, generated from the unmodified reference build by
tests/golden/make_ref_symbols.py) -- that is what "src/training links against it unchanged" means at the ABI level."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libgsplat_backend_b200.so")


def test_reference_symbol_fixture_is_complete():
    names = open(os.path.join(ROOT, "tests", "golden", "ref_symbols.txt")).read().split()
    demangled = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout
    for fn in ("spherical_harmonics_fwd", "spherical_harmonics_bwd", "intersect_tile", "intersect_offset",
               "quats_to_rotmats", "relocation", "add_noise", "projection_ut_3dgs_fused",
               "rasterize_to_pixels_from_world_3dgs_fwd", "rasterize_to_pixels_from_world_3dgs_bwd"):
        assert f"gsplat::{fn}(" in demangled
    assert "fast_gs::optimizer::adam_step(" in demangled
    assert "fast_gs::rasterization::forward_wrapper(" in demangled
    assert "fast_gs::rasterization::backward_wrapper(" in demangled


def test_host_layer_exports_the_reference_symbols():
    if not os.path.exists(LIB):
        pytest.skip("host layer not built (needs the reference headers: make -C lichtfeld-studio_b200/host)")
    out = subprocess.run(["nm", "-D", "--defined-only", LIB], capture_output=True, text=True).stdout
    mine = {l.split()[-1] for l in out.splitlines() if l.strip()}
    want = set(open(os.path.join(ROOT, "tests", "golden", "ref_symbols.txt")).read().split())
    missing = sorted(want - mine)
    assert not missing, missing
    assert "_ZN7fast_gs9optimizer17adam_step_wrapperERN2at6TensorES3_S3_RKS2_ffffff" in mine
