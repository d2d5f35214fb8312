"""ctypes binding of libgsicp_b200.so (the C ABI declared in include/gsicp_b200.h).

The CUDA library is the product: there is NO CPU or PyTorch fallback.  Importing this module
raises ImportError when the shared library has not been built
(`python -c "import __graft_entry__ as g; g.build()"` or `make -C gs_icp_slam_b200/csrc`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgsicp_b200.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build the sm_100a CUDA library first "
        "(make -C gs_icp_slam_b200/csrc). gs_icp_slam_b200 has no CPU fallback."
    )

lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)

ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_size_t, C.c_void_p)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p)
ALLREDUCE_F32_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p)


class RasterArgs(C.Structure):
    """struct gsicp_raster_args (include/gsicp_b200.h)."""

    _fields_ = [
        ("P", C.c_int),
        ("D", C.c_int),
        ("M", C.c_int),
        ("width", C.c_int),
        ("height", C.c_int),
        ("tan_fovx", C.c_float),
        ("tan_fovy", C.c_float),
        ("scale_modifier", C.c_float),
        ("prefiltered", C.c_int),
        ("debug", C.c_int),
        ("d_background", C.c_void_p),
        ("d_means3D", C.c_void_p),
        ("d_shs", C.c_void_p),
        ("d_colors_precomp", C.c_void_p),
        ("d_opacities", C.c_void_p),
        ("d_scales", C.c_void_p),
        ("d_rotations", C.c_void_p),
        ("d_cov3D_precomp", C.c_void_p),
        ("d_viewmatrix", C.c_void_p),
        ("d_projmatrix", C.c_void_p),
        ("d_campos", C.c_void_p),
        ("tile_shard_count", C.c_int),
        ("tile_shard_index", C.c_int),
    ]


BOUND = []


def _sig(name, restype, argtypes):
    fn = getattr(lib, name)  # AttributeError here = the library does not export what the header declares
    BOUND.append(name)
    fn.restype = restype
    fn.argtypes = argtypes
    return fn


vp, i32, f64p = C.c_void_p, C.c_int, C.POINTER(C.c_double)

_sig("gsicp_last_error", C.c_char_p, [])
_sig("gsicp_build_info", C.c_char_p, [])
_sig("gsicp_launch_count", C.c_uint64, [])

_sig("gsicp_prof_enable", None, [i32])
_sig("gsicp_prof_reset", None, [])
_sig("gsicp_prof_count", i32, [])
_sig("gsicp_prof_name", C.c_char_p, [i32])
_sig("gsicp_prof_read", i32, [i32, f64p, C.POINTER(C.c_long)])

_sig("gsicp_raster_forward", i32, [C.POINTER(RasterArgs), vp, vp, vp, vp, ALLOC_FN, ALLOC_FN, ALLOC_FN, vp, vp])
_sig("gsicp_raster_backward_work_bytes", C.c_size_t, [i32])
_sig("gsicp_raster_set_allreduce", i32, [ALLREDUCE_F32_FN, vp])
_sig("gsicp_raster_backward", i32, [C.POINTER(RasterArgs), i32, vp, vp, vp, vp, vp, vp] + [vp] * 8 + [vp, vp])
_sig("gsicp_raster_export_binning", i32, [C.POINTER(RasterArgs), i32, vp, vp, vp, vp, vp])
_sig("gsicp_mark_visible", i32, [i32, vp, vp, vp, vp, vp])
_sig("gsicp_test_set_render_cull", None, [i32])
_sig("gsicp_test_set_bwd_variant", None, [i32])
_sig("gsicp_test_preload_kernels", i32, [])
_sig("gsicp_dist2", i32, [i32, vp, vp, vp])

_sig("gsicp_gicp_create", vp, [])
_sig("gsicp_gicp_destroy", None, [vp])
_sig("gsicp_gicp_set_max_correspondence_distance", i32, [vp, C.c_double])
_sig("gsicp_gicp_set_max_knn_distance", i32, [vp, C.c_double])
_sig("gsicp_gicp_set_correspondence_randomness", i32, [vp, i32])
_sig("gsicp_gicp_set_max_iterations", i32, [vp, i32])
for _n in ("source", "target"):
    _sig(f"gsicp_gicp_set_input_{_n}", i32, [vp, vp, i32, i32])
    _sig(f"gsicp_gicp_set_input_{_n}_device", i32, [vp, vp, i32])
    _sig(f"gsicp_gicp_set_{_n}_filter", i32, [vp, i32, vp, i32])
    _sig(f"gsicp_gicp_set_{_n}_covariances_fromqs", i32, [vp, vp, vp, i32])
    _sig(f"gsicp_gicp_set_{_n}_covariances_fromqs_device", i32, [vp, vp, vp, i32])
    _sig(f"gsicp_gicp_{_n}_size", i32, [vp])
    _sig(f"gsicp_gicp_{_n}_rotationsq_size", i32, [vp])
    _sig(f"gsicp_gicp_{_n}_scales_size", i32, [vp])
    _sig(f"gsicp_gicp_get_{_n}_rotationsq", i32, [vp, vp])
    _sig(f"gsicp_gicp_get_{_n}_scales", i32, [vp, vp])
    _sig(f"gsicp_gicp_get_{_n}_covariances", i32, [vp, vp])
_sig("gsicp_gicp_calculate_target_covariance_with_filter", i32, [vp])
_sig("gsicp_gicp_calculate_source_covariance", i32, [vp])
_sig("gsicp_gicp_calculate_target_covariance", i32, [vp])
_sig("gsicp_gicp_calculate_target_covariance_withz", i32, [vp])
_sig("gsicp_gicp_set_source_z_values", i32, [vp, vp, i32])
_sig("gsicp_gicp_set_target_z_values", i32, [vp, vp, i32])
_sig("gsicp_gicp_swap_source_and_target", i32, [vp])
_sig("gsicp_gicp_get_fitness_score", i32, [vp, C.c_double, vp])
_sig("gsicp_gicp_align", i32, [vp, vp, vp])
_sig("gsicp_gicp_has_converged", i32, [vp])
_sig("gsicp_gicp_get_final_hessian", i32, [vp, vp])
_sig("gsicp_gicp_get_source_correspondence", i32, [vp, vp, vp])
_sig("gsicp_gicp_linearize", i32, [vp, vp, vp, vp, vp])
_sig("gsicp_gicp_compute_error", i32, [vp, vp, vp])
_sig("gsicp_gicp_set_shard", i32, [vp, i32, i32, ALLREDUCE_FN, vp])
_sig("gsicp_gicp_set_stream", i32, [vp, vp])
_sig("gsicp_gicp_set_host_lm", i32, [vp, i32])
_sig("gsicp_gicp_set_source_filter_device", i32, [vp, i32, vp, i32])
_sig("gsicp_gicp_set_target_filter_device", i32, [vp, i32, vp, i32])
_sig("gsicp_comm_alloc", i32, [C.c_size_t, C.POINTER(vp), vp])
_sig("gsicp_comm_connect", i32, [vp, i32, i32, vp])
_sig("gsicp_comm_connect_local", i32, [vp, i32, i32, C.POINTER(vp)])
_sig("gsicp_comm_destroy", None, [vp])
_sig("gsicp_comm_world", i32, [vp])
_sig("gsicp_comm_rank", i32, [vp])
_sig("gsicp_comm_barrier", i32, [vp, vp])
_sig("gsicp_gicp_set_comm", i32, [vp, vp])
_sig("gsicp_raster_set_comm", i32, [vp])
_sig("gsicp_mapping_loss_work_bytes", C.c_size_t, [i32, i32])
_sig("gsicp_mapping_loss_forward", i32, [i32, i32, vp, vp, vp, vp, C.c_float, C.c_float, C.c_float, i32, vp, vp, vp, vp, vp])
_sig("gsicp_mapping_loss_backward", i32, [i32, i32, vp, vp, vp, vp, C.c_float, C.c_float, C.c_float, i32, vp, vp, vp, vp, vp])

# BOUND lists every bound symbol; tests/test_abi.py checks include/gsicp_b200.h against it.


class GsicpError(RuntimeError):
    pass


def check(rc, what="libgsicp_b200"):
    """Raise on a negative status (the ABI's error convention); return rc otherwise."""
    if rc is not None and rc < 0:
        msg = lib.gsicp_last_error().decode("utf-8", "replace")
        raise GsicpError(f"{what} failed ({rc}): {msg}")
    return rc


def last_error():
    return lib.gsicp_last_error().decode("utf-8", "replace")


def build_info():
    return lib.gsicp_build_info().decode()


def launch_count():
    return int(lib.gsicp_launch_count())


def prof_enable(on=True):
    lib.gsicp_prof_enable(1 if on else 0)


def prof_reset():
    lib.gsicp_prof_reset()


def prof_read():
    """{kernel name: (total_ms, launches)} accumulated since the last reset (device time, CUDA events)."""
    out = {}
    for k in range(lib.gsicp_prof_count()):
        ms, n = C.c_double(0), C.c_long(0)
        lib.gsicp_prof_read(k, C.byref(ms), C.byref(n))
        out[lib.gsicp_prof_name(k).decode()] = (ms.value, n.value)
    return out
