"""ctypes binding of libnrt_b200.so (C ABI: include/nrt_b200.h).

There is no fallback: if the library is missing or a call fails, an exception is raised."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_TAG = os.environ.get("NRT_LIB_TAG", "")   # development: a kernel variant built with NRT_BUILD_TAG (build_native.py)
LIB_PATH = os.path.join(_HERE, "lib", "libnrt_b200%s.so" % ("_" + _TAG if _TAG else ""))

OK, E_INVALID, E_CUDA, E_UNSUPPORTED = 0, -1, -2, -3
ACT_LEAKY_RELU, ACT_SOFTPLUS = 0, 1
OUT_NONE, OUT_SIGMOID, OUT_SOFTPLUS, OUT_TANH = 0, 1, 2, 3
PREC_F32, PREC_F16, PREC_BF16 = 0, 1, 2
MAX_LAYERS = 20
MAX_HIER_SAMPLES = 512     # NRT_MAX_HIER_SAMPLES: n_coarse + n_fine the merge kernels hold in shared memory

c_int, c_i64, c_f32, c_f64, c_vp, c_sz = (ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_double,
                                          ctypes.c_void_p, ctypes.c_size_t)


class NrtMlp(ctypes.Structure):
    _fields_ = [("in_size", ctypes.c_int32), ("latent_size", ctypes.c_int32), ("freqs", ctypes.c_int32),
                ("hidden", ctypes.c_int32), ("num_layers", ctypes.c_int32), ("skip", ctypes.c_int32),
                ("out_size", ctypes.c_int32), ("act", ctypes.c_int32),
                ("basis", c_vp), ("params", c_vp), ("params_tc", c_vp)]


class NrtSphereSdf(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int32), ("centers", c_vp), ("radii", c_vp), ("tfs", c_vp), ("shift", NrtMlp)]


class NrtNerfSampling(ctypes.Structure):
    _fields_ = [("n_coarse", ctypes.c_int32), ("n_fine", ctypes.c_int32), ("t_near", c_f32), ("t_far", c_f32),
                ("jitter_seed", ctypes.c_uint64)]


class NrtCamera(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("n_views", ctypes.c_int32), ("a", c_vp), ("b", c_vp),
                ("a_view_stride", ctypes.c_int32), ("a_row_stride", ctypes.c_int32),
                ("b_view_stride", ctypes.c_int32), ("b_row_stride", ctypes.c_int32),
                ("focal", c_f32), ("size", c_f32), ("x0", ctypes.c_int32), ("y0", ctypes.c_int32),
                ("nx", ctypes.c_int32), ("ny", ctypes.c_int32), ("bundle", ctypes.c_int32),
                ("pos_per_pixel", ctypes.c_int32), ("positions", c_vp), ("jitter", c_f32),
                ("jitter_seed", ctypes.c_uint64)]


MAX_BSDFS = 16
MAX_LATTICE_DIM = 1024     # NRT_MAX_LATTICE_DIM


class NrtLattice(ctypes.Structure):
    _fields_ = [("nx", c_i64), ("ny", c_i64), ("nz", c_i64), ("origin", c_f32 * 3), ("spacing", c_f32 * 3)]


class NrtOccupancy(ctypes.Structure):
    _fields_ = [("res", ctypes.c_int32), ("bbox_min", c_f32 * 3), ("bbox_max", c_f32 * 3), ("bits", c_vp)]


class NrtLight(ctypes.Structure):
    _fields_ = [("mode", ctypes.c_int32), ("n_views", ctypes.c_int32), ("location", c_vp), ("amp", c_vp), ("coef", c_vp),
                ("view_of_hit", c_vp), ("v", c_vp), ("sig_color", c_vp)]


class NrtBlend(ctypes.Structure):
    _fields_ = [("nb", ctypes.c_int32), ("kind", ctypes.c_int32 * MAX_BSDFS), ("neural_act", ctypes.c_int32),
                ("diffuse_pre", ctypes.c_int32)]


class NrtError(RuntimeError):
    pass


_PM, _PS, _PN = ctypes.POINTER(NrtMlp), ctypes.POINTER(NrtSphereSdf), ctypes.POINTER(NrtNerfSampling)
_PL, _PB = ctypes.POINTER(NrtLight), ctypes.POINTER(NrtBlend)
_PC = ctypes.POINTER(NrtCamera)
_PG = ctypes.POINTER(NrtLattice)
_PO = ctypes.POINTER(NrtOccupancy)

# every symbol declared in include/nrt_b200.h: name -> (restype, argtypes)
SIGNATURES = {
    "nrt_abi_version": (c_int, []),
    "nrt_last_error": (ctypes.c_char_p, []),
    "nrt_device_info": (c_int, [ctypes.POINTER(c_int)] * 3),
    "nrt_profile_enable": (c_int, [c_int]),
    "nrt_profile_num_tags": (c_int, []),
    "nrt_profile_tag_name": (ctypes.c_char_p, [c_int]),
    "nrt_profile_collect": (c_int, [c_int, ctypes.POINTER(c_f64), ctypes.POINTER(ctypes.c_longlong)]),
    "nrt_mlp_param_count": (c_i64, [_PM]),
    "nrt_mlp_tc_blob_bytes": (c_i64, [_PM, c_int]),
    "nrt_mlp_pack_tc": (c_int, [_PM, c_int, c_vp, c_vp]),
    "nrt_mlp_forward": (c_int, [_PM, c_int, c_int, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "nrt_mlp_backward": (c_int, [_PM, c_int, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nrt_mlp_train_tc_workspace_bytes": (c_i64, [_PM, c_i64]),
    "nrt_mlp_tc_dgrad_blob_bytes": (c_i64, [_PM, c_int]),
    "nrt_mlp_pack_tc_dgrad": (c_int, [_PM, c_int, c_int, c_vp, c_vp]),
    "nrt_mlp_forward_train_tc": (c_int, [_PM, c_int, c_int, c_vp, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "nrt_mlp_backward_tc": (c_int, [_PM, c_int, c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp, c_vp, c_vp]),
    "nrt_nerfle_train_forward": (c_int, [_PM, _PM, c_int, c_vp, c_i64, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp,
                                         c_vp, c_sz, c_vp, c_sz, c_vp]),
    "nrt_nerfle_train_forward_ts": (c_int, [_PM, _PM, c_int, c_vp, c_i64, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp,
                                            c_vp, c_sz, c_vp, c_sz, c_vp]),
    "nrt_nerfle_train_backward": (c_int, [_PM, _PM, c_int, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                          c_vp, c_vp, c_vp, c_vp]),
    "nrt_sdf_eval": (c_int, [_PS, c_int, c_vp, c_i64, c_vp, c_vp]),
    "nrt_sdf_value_grad": (c_int, [_PS, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "nrt_sphere_set_forward": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "nrt_sphere_set_backward": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nrt_mlp_value_jac_forward": (c_int, [_PM, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "nrt_mlp_value_jac_backward": (c_int, [_PM, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nrt_mlp_value_jac_tc_workspace_bytes": (c_i64, [_PM, c_i64]),
    "nrt_mlp_value_jac_forward_tc": (c_int, [_PM, c_int, c_vp, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "nrt_mlp_value_jac_backward_tc": (c_int, [_PM, c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp, c_vp]),
    "nrt_sdf_sphere_trace": (c_int, [_PS, c_int, c_vp, c_vp, c_i64, c_f32, c_int, c_f32, c_vp, c_vp, c_vp, c_vp]),
    "nrt_sdf_shadow_test": (c_int, [_PS, c_int, c_vp, c_vp, c_vp, c_i64, c_f32, c_int, c_vp, c_vp, c_vp]),
    "nrt_sdf_min_scan": (c_int, [_PS, c_int, c_vp, c_i64, c_f64, c_int, c_vp, c_vp, c_vp, c_vp]),
    "nrt_composite_forward": (c_int, [c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_vp]),
    "nrt_composite_backward": (c_int, [c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "nrt_composite_forward_ts": (c_int, [c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_vp]),
    "nrt_composite_backward_ts": (c_int, [c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "nrt_nerfle_render": (c_int, [_PM, _PM, c_int, c_vp, c_i64, c_vp, _PN, c_vp, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "nrt_nerfle_render_workspace": (c_sz, [_PM, _PM, c_int, c_i64, _PN]),
    "nrt_nerfle_sample_hierarchical_workspace": (c_sz, [_PM, _PM, c_int, c_i64, _PN]),
    "nrt_nerfle_sample_hierarchical": (c_int, [_PM, _PM, c_int, c_vp, c_i64, _PN, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_sz,
                                               c_vp]),
    "nrt_nerfle_render_host": (c_int, [_PM, _PM, c_int, c_vp, c_i64, c_vp, c_int, _PN, c_vp, c_int, c_vp, c_vp]),
    "nrt_camera_rays": (c_int, [_PC, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "nrt_set_camera_rays_mode": (c_int, [c_int]),
    "nrt_nerfle_render_camera_workspace": (c_sz, [_PM, _PM, c_int, _PC, _PN]),
    "nrt_nerfle_render_camera": (c_int, [_PM, _PM, c_int, _PC, c_vp, _PN, c_vp, c_int, c_vp, c_vp, c_sz, c_vp]),
    "nrt_nerfle_render_samples_workspace": (c_sz, [_PM, _PM, c_int, c_i64, c_int, _PC]),
    "nrt_nerfle_render_samples": (c_int, [_PM, _PM, c_int, c_vp, _PC, c_i64, c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp,
                                          c_vp, c_sz, c_vp]),
    "nrt_nerfle_render_camera_host":(c_int, [_PM, _PM, c_int, _PC, c_vp, c_int, _PN, c_vp, c_int, c_vp, c_vp]),
    "nrt_occupancy_update_workspace": (c_sz, [_PM, c_int, ctypes.c_int32, c_int]),
    "nrt_occupancy_update": (c_int, [_PM, c_int, _PO, c_int, c_f32, c_f32, ctypes.c_uint64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "nrt_occupancy_mask": (c_int, [_PO, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_vp]),
    "nrt_nerfle_render_occupancy_workspace": (c_sz, [_PM, _PM, c_int, c_i64, _PC, _PN]),
    "nrt_nerfle_render_occupancy": (c_int, [_PM, _PM, c_int, c_vp, _PC, c_i64, c_vp, _PN, c_vp, c_int, c_vp, _PO, c_vp, c_vp,
                                            c_vp, c_sz, c_vp]),
    "nrt_nerfle_render_samples_occupancy_workspace": (c_sz, [_PM, _PM, c_int, c_i64, c_int, _PC]),
    "nrt_nerfle_render_samples_occupancy": (c_int, [_PM, _PM, c_int, c_vp, _PC, c_i64, c_vp, c_vp, c_int, c_vp, c_int, c_vp,
                                                    _PO, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "nrt_sdf_lattice_eval_workspace": (c_i64, [_PG]),
    "nrt_sdf_lattice_eval": (c_int, [_PS, c_int, _PG, c_vp, c_vp, c_sz, c_vp]),
    "nrt_isosurface_workspace": (c_i64, [_PG]),
    "nrt_isosurface_count": (c_int, [_PG, c_vp, c_f32, c_vp, c_sz, c_vp, c_vp]),
    "nrt_isosurface_emit": (c_int, [_PG, c_vp, c_f32, c_vp, c_sz, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "nrt_shading_frame": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "nrt_to_local": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp]),
    "nrt_param_rusin2": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp]),
    "nrt_shade_geom_forward": (c_int, [c_vp, c_vp, c_vp, c_i64, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nrt_shade_geom_backward": (c_int, [c_vp, c_vp, c_i64, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nrt_shade_light_forward": (c_int, [_PL, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nrt_shade_light_backward": (c_int, [_PL, c_vp, c_vp, c_vp, c_i64] + [c_vp] * 11),
    "nrt_shade_blend_forward": (c_int, [_PB] + [c_vp] * 8 + [c_f32, c_i64, c_vp, c_vp]),
    "nrt_shade_blend_backward": (c_int, [_PB] + [c_vp] * 8 + [c_f32, c_i64] + [c_vp] * 10),
}

_lib = None


def lib():
    """Loads libnrt_b200.so; raises (never falls back) if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NrtError("libnrt_b200.so not built at %s -- run `python -c 'import __graft_entry__ as g; "
                           "g.build()'` (needs nvcc); there is no CPU/PyTorch fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)      # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        if L.nrt_abi_version() != 1:
            raise NrtError("libnrt_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        msg = lib().nrt_last_error().decode("utf-8", "replace")
        raise NrtError("libnrt_b200 call failed (%d): %s" % (rc, msg))
