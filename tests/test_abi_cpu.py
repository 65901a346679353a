"""CPU-side checks of the C-ABI library: it loads without a GPU, exports every symbol that
include/nrt_b200.h declares, validates descriptors, and fails loudly (no fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "nrt_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(nrt_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    from neural_raytracing_b200 import _native
    L = _native.lib()
    syms = _declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), "libnrt_b200.so does not export %s" % s
        assert s in _native.SIGNATURES, "binding missing for %s" % s
    assert sorted(_native.SIGNATURES) == syms


def test_param_count_matches_reference_shapes():
    from neural_raytracing_b200 import _native as N
    # SURVEY.md section 8 catalogue (verified against the instantiated reference)
    cases = {
        (3, 0, 32, 128, 8, 3, 1): 166657,     # SphereSDF.shift
        (3, 0, 64, 96, 6, 3, 3): 93987,       # NeuralBSDF.mlp
        (5, 0, 16, 64, 8, 3, 1): 42881,       # occlusion MLP
        (3, 0, 16, 256, 10, 3, 3): 694787,    # LightField
        (3, 0, 16, 128, 5, 3, 65): 104513,    # NeRFLE.first
        (70, 0, 16, 64, 8, 3, 3): 59651,      # NeRFLE.second (PT)
        (115, 0, 16, 64, 8, 3, 3): 71171,     # NeRFLE.second (LE)
        (3, 0, 128, 256, 16, 3, 4): 1451780,  # sp_var_fn nb=4
    }
    for (i, lat, f, h, L, sk, o), n in cases.items():
        m = N.NrtMlp(i, lat, f, h, L, sk, o, 0, None, None, None)
        assert N.lib().nrt_mlp_param_count(ctypes.byref(m)) == n


def test_compute_call_without_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from neural_raytracing_b200 import _native as N
    rc = N.lib().nrt_device_info(None, None, None)
    assert rc == N.E_CUDA
    with pytest.raises(N.NrtError):
        N.check(rc)


def test_ops_reject_cpu_tensors_no_fallback():
    import torch
    from neural_raytracing_b200 import ops
    with pytest.raises(ops.NrtError):
        ops.composite_forward(torch.zeros(4, 2), torch.zeros(4, 2, 3), torch.zeros(4))


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under neural_raytracing_b200/ may reference it."""
    pkg = os.path.join(ROOT, "neural_raytracing_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), fn
                assert "nrt_oracle" not in txt.replace("oracle/c/nrt_oracle.c", ""), fn


def test_render_samples_export_and_argument_checks():
    """nrt_nerfle_render_samples is exported and rejects malformed calls before touching a device"""
    import ctypes as C
    from neural_raytracing_b200 import _native as N
    L = N.lib()
    assert "nrt_nerfle_render_samples" in _declared_symbols()
    assert "nrt_nerfle_render_samples_workspace" in _declared_symbols()
    m = N.NrtMlp(3, 0, 16, 128, 5, 3, 65, 0, None, None, None)
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)

    def call(rays, cam, R, ts, ts_pr, S, sig=p, rgb=p):
        return L.nrt_nerfle_render_samples(C.byref(m), C.byref(m), N.PREC_F16, rays, cam, R, ts, ts_pr, S, p, 3, None,
                                           sig, rgb, p, 256, None)
    cases = [((None, None, 4, p, None, 8), "exactly one of rays / cam"),
             ((p, None, -1, p, None, 8), "negative R"),
             ((p, None, 4, p, p, 8), "exactly one of ts / ts_per_ray"),
             ((p, None, 4, None, None, 8), "exactly one of ts / ts_per_ray"),
             ((p, None, 4, p, None, 0), "bad sample count")]
    for args, msg in cases:
        assert call(*args) == N.E_INVALID
        assert msg in L.nrt_last_error().decode(), L.nrt_last_error()
    assert call(p, None, 4, p, None, 8, sig=None) == N.E_INVALID
    assert "null out_sigma/out_rgb" in L.nrt_last_error().decode()
    cam = N.NrtCamera()                 # NRT_CAM_NERF with no views: validated as the camera render validates it
    assert call(None, C.byref(cam), 4, p, None, 8) == N.E_INVALID
    assert "bad block" in L.nrt_last_error().decode()
