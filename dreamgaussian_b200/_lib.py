"""ctypes binding of libdgr_b200.so (the C ABI declared in include/dgr_b200.h).

There is NO fallback: if the shared library is missing or does not load, importing the compute entry points raises.
The library is built in-tree by ``dreamgaussian_b200.build`` (nvcc, sm_100a).
"""
import ctypes
import os

from . import build as _build

c_f32p = ctypes.c_void_p  # device pointers travel as integers
ABI_VERSION = 4          # include/dgr_b200.h DGR_ABI_VERSION


class DgrSettings(ctypes.Structure):
    _fields_ = [
        ("image_height", ctypes.c_int32), ("image_width", ctypes.c_int32),
        ("tanfovx", ctypes.c_float), ("tanfovy", ctypes.c_float), ("scale_modifier", ctypes.c_float),
        ("sh_degree", ctypes.c_int32), ("prefiltered", ctypes.c_int32), ("debug", ctypes.c_int32),
        ("bg", c_f32p), ("viewmatrix", c_f32p), ("projmatrix", c_f32p), ("campos", c_f32p),
    ]


class DgrGaussians(ctypes.Structure):
    _fields_ = [
        ("P", ctypes.c_int32), ("M", ctypes.c_int32),
        ("means3D", c_f32p), ("shs", c_f32p), ("colors_precomp", c_f32p), ("opacities", c_f32p),
        ("scales", c_f32p), ("rotations", c_f32p), ("cov3D_precomp", c_f32p),
        ("shs_rest", c_f32p), ("activations", ctypes.c_int32),          # raw GaussianModel parameters (SURVEY §8 f1)
    ]


class DgrAdamGroup(ctypes.Structure):
    _fields_ = [("param", c_f32p), ("grad", c_f32p), ("exp_avg", c_f32p), ("exp_avg_sq", c_f32p), ("n", ctypes.c_uint64),
                ("lr", ctypes.c_float), ("step", ctypes.c_int32)]


class DgrDensifyTensors(ctypes.Structure):
    _fields_ = [("inp", c_f32p * 6), ("exp_avg_in", c_f32p * 6), ("exp_avg_sq_in", c_f32p * 6),
                ("out", c_f32p * 6), ("exp_avg_out", c_f32p * 6), ("exp_avg_sq_out", c_f32p * 6), ("width", ctypes.c_int32 * 6)]


class DgrImages(ctypes.Structure):
    _fields_ = [("color", c_f32p), ("depth", c_f32p), ("alpha", c_f32p), ("radii", ctypes.c_void_p)]


class DgrImageGrads(ctypes.Structure):
    _fields_ = [("dL_dcolor", c_f32p), ("dL_ddepth", c_f32p), ("dL_dalpha", c_f32p)]


class DgrGaussianGrads(ctypes.Structure):
    _fields_ = [
        ("dL_dmeans3D", c_f32p), ("dL_dmeans2D", c_f32p), ("dL_dshs", c_f32p), ("dL_dcolors_precomp", c_f32p),
        ("dL_dopacities", c_f32p), ("dL_dscales", c_f32p), ("dL_drotations", c_f32p), ("dL_dcov3D_precomp", c_f32p),
        ("accumulate", ctypes.c_int32),
        ("dL_dshs_rest", c_f32p), ("xyz_gradient_accum", c_f32p), ("denom", c_f32p), ("max_radii2D", c_f32p),
        ("push", ctypes.c_void_p),
    ]


class DgrPeerPush(ctypes.Structure):
    _fields_ = [("world", ctypes.c_int32), ("rank", ctypes.c_int32), ("gaussians_per_owner", ctypes.c_int64),
                ("delta_floats", ctypes.c_int64 * 16)]


EXPORTS = (
    "dgr_abi_version", "dgr_last_error", "dgr_launch_count", "dgr_reset_launch_count",
    "dgr_geom_bytes", "dgr_image_bytes", "dgr_binning_bytes",
    "dgr_forward_preprocess", "dgr_forward_render", "dgr_backward", "dgr_mark_visible", "dgr_debug_geom",
    "dgr_profile_enable", "dgr_profile_collect", "dgr_event_create", "dgr_event_synchronize", "dgr_event_destroy", "dgr_set_tuning", "dgr_peer_allreduce", "dgr_peer_flag_bytes", "dgr_peer_reduce_staged", "dgr_peer_push_flat", "dgr_knn_scratch_bytes", "dgr_dist_cuda2", "dgr_fields_scratch_bytes", "dgr_extract_fields", "dgr_adam_step", "dgr_densify_scratch_bytes", "dgr_densify_plan", "dgr_densify_apply",
    "dgr_batch_geom_bytes", "dgr_batch_image_bytes", "dgr_forward_preprocess_batch", "dgr_backward_batch",
)

_lib = None


def library_path():
    return _build.LIB_PATH


def load():
    """Load libdgr_b200.so (building it first if nvcc is available and the sources are newer). Raises on failure."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if _build.is_stale():
        try:
            _build.build()
        except Exception as e:  # no nvcc on this machine and no prebuilt library: nothing to fall back to
            if not os.path.exists(path):
                raise RuntimeError(
                    "libdgr_b200.so is not built and could not be compiled here (%s). "
                    "Run `python -m dreamgaussian_b200.build` on a machine with nvcc." % e)
    lib = ctypes.CDLL(path)
    vp, u64, i32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32
    lib.dgr_abi_version.restype = ctypes.c_int
    lib.dgr_last_error.restype = ctypes.c_char_p
    lib.dgr_launch_count.restype = u64
    lib.dgr_reset_launch_count.restype = None
    lib.dgr_geom_bytes.restype = ctypes.c_size_t
    lib.dgr_geom_bytes.argtypes = [i32, i32, i32]
    lib.dgr_image_bytes.restype = ctypes.c_size_t
    lib.dgr_image_bytes.argtypes = [i32, i32]
    lib.dgr_binning_bytes.restype = ctypes.c_size_t
    lib.dgr_binning_bytes.argtypes = [u64, i32, i32]
    lib.dgr_forward_preprocess.restype = ctypes.c_int
    lib.dgr_forward_preprocess.argtypes = [ctypes.POINTER(DgrSettings), ctypes.POINTER(DgrGaussians), vp, vp, vp, vp]
    lib.dgr_batch_geom_bytes.restype = ctypes.c_size_t
    lib.dgr_batch_geom_bytes.argtypes = [i32, i32, i32, i32]
    lib.dgr_batch_image_bytes.restype = ctypes.c_size_t
    lib.dgr_batch_image_bytes.argtypes = [i32, i32, i32]
    lib.dgr_forward_preprocess_batch.restype = ctypes.c_int        # settings: a ctypes array of V DgrSettings
    lib.dgr_forward_preprocess_batch.argtypes = [vp, i32, ctypes.POINTER(DgrGaussians), vp, vp, vp, vp]
    lib.dgr_backward_batch.restype = ctypes.c_int                  # settings / binning / capacities / gin: host arrays of V
    lib.dgr_backward_batch.argtypes = [vp, i32, ctypes.POINTER(DgrGaussians), vp, vp, vp, vp, vp, vp, ctypes.POINTER(DgrGaussianGrads), vp]
    lib.dgr_peer_allreduce.restype = ctypes.c_int
    lib.dgr_peer_allreduce.argtypes = [vp, i32, i32, u64, u64, vp, ctypes.c_uint32, vp]
    lib.dgr_peer_reduce_staged.restype = ctypes.c_int
    lib.dgr_peer_reduce_staged.argtypes = [vp, vp, ctypes.c_int64, i32, vp, vp, u64, u64, u64, vp, ctypes.c_uint32, vp]
    lib.dgr_peer_push_flat.restype = ctypes.c_int
    lib.dgr_peer_push_flat.argtypes = [vp, vp, ctypes.c_int64, i32, vp, vp, vp]
    lib.dgr_peer_flag_bytes.restype = ctypes.c_size_t
    lib.dgr_set_tuning.restype = ctypes.c_int
    lib.dgr_set_tuning.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.dgr_event_create.restype = vp
    lib.dgr_event_synchronize.restype = ctypes.c_int
    lib.dgr_event_synchronize.argtypes = [vp]
    lib.dgr_event_destroy.restype = None
    lib.dgr_event_destroy.argtypes = [vp]
    lib.dgr_forward_render.restype = ctypes.c_int
    lib.dgr_forward_render.argtypes = [ctypes.POINTER(DgrSettings), ctypes.POINTER(DgrGaussians), vp, vp, u64, vp,
                                       ctypes.POINTER(DgrImages), i32, vp, u64, vp, vp]
    lib.dgr_backward.restype = ctypes.c_int
    lib.dgr_backward.argtypes = [ctypes.POINTER(DgrSettings), ctypes.POINTER(DgrGaussians), vp, vp, u64, vp, vp, vp,
                                 ctypes.POINTER(DgrImageGrads), ctypes.POINTER(DgrGaussianGrads), vp]
    lib.dgr_knn_scratch_bytes.restype = ctypes.c_size_t
    lib.dgr_knn_scratch_bytes.argtypes = [i32]
    lib.dgr_dist_cuda2.restype = ctypes.c_int
    lib.dgr_dist_cuda2.argtypes = [i32, vp, vp, vp, vp]
    lib.dgr_fields_scratch_bytes.restype = ctypes.c_size_t
    lib.dgr_fields_scratch_bytes.argtypes = [i32, i32]
    lib.dgr_extract_fields.restype = ctypes.c_int
    lib.dgr_extract_fields.argtypes = [i32, vp, vp, vp, vp, i32, i32, ctypes.c_float, vp, vp, vp, vp]
    lib.dgr_adam_step.restype = ctypes.c_int
    lib.dgr_adam_step.argtypes = [ctypes.POINTER(DgrAdamGroup), i32, ctypes.c_double, ctypes.c_double, ctypes.c_double, vp]
    lib.dgr_densify_scratch_bytes.restype = ctypes.c_size_t
    lib.dgr_densify_scratch_bytes.argtypes = [i32]
    lib.dgr_densify_plan.restype = ctypes.c_int
    lib.dgr_densify_plan.argtypes = [i32, vp, vp, vp, vp, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, i32, vp, vp, vp]
    lib.dgr_densify_apply.restype = ctypes.c_int
    lib.dgr_densify_apply.argtypes = [i32, ctypes.POINTER(DgrDensifyTensors), vp, vp, vp]
    lib.dgr_mark_visible.restype = ctypes.c_int
    lib.dgr_mark_visible.argtypes = [i32, vp, vp, vp, vp, vp]
    lib.dgr_debug_geom.restype = ctypes.c_int
    lib.dgr_debug_geom.argtypes = [i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.dgr_profile_enable.restype = None
    lib.dgr_profile_enable.argtypes = [ctypes.c_int]
    lib.dgr_profile_collect.restype = ctypes.c_int
    lib.dgr_profile_collect.argtypes = [ctypes.c_char_p, ctypes.c_size_t, vp, ctypes.c_int]
    if lib.dgr_abi_version() != ABI_VERSION:
        raise RuntimeError("libdgr_b200.so ABI version mismatch")
    _lib = lib
    tune = os.environ.get("DGR_TUNING")        # "ppl_fwd,ppl_bwd,tile_order" for experiments
    if tune:
        a, b, c = (int(x) for x in tune.split(","))
        check(lib.dgr_set_tuning(a, b, c))
    return lib


def profile_collect(max_records=4096):
    """-> list of (kernel name, milliseconds) recorded since dgr_profile_enable(1)."""
    lib = load()
    names = ctypes.create_string_buffer(64 * max_records)
    ms = (ctypes.c_float * max_records)()
    n = lib.dgr_profile_collect(names, len(names), ctypes.cast(ms, ctypes.c_void_p), max_records)
    nm = names.value.decode().split("\n")[:n]
    return list(zip(nm, [float(ms[i]) for i in range(n)]))


def check(code):
    if code != 0:
        raise RuntimeError("libdgr_b200: %s (code %d)" % (load().dgr_last_error().decode(), code))
