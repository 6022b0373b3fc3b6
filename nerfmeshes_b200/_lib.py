"""ctypes binding of libnerfmeshes_b200.so — the stub a reference-side maintainer would add (INTEGRATION.md).

No torch types cross this boundary: pointers are integers (tensor.data_ptr()), sizes are ints.  There is no CPU
fallback anywhere above this file: if the shared library is missing, loading fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libnerfmeshes_b200.so")


class NmNetDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "num_layers", "hidden_size", "skip_step", "num_encoding_fn_xyz", "num_encoding_fn_dir",
        "include_input_xyz", "include_input_dir", "log_sampling_xyz", "log_sampling_dir", "use_viewdirs")]


class NmRenderCfg(C.Structure):
    _fields_ = [("num_coarse", C.c_int32), ("num_fine", C.c_int32), ("lindisp", C.c_int32), ("perturb", C.c_int32),
                ("white_background", C.c_int32), ("noise_std", C.c_float), ("attenuation_threshold", C.c_float),
                ("precision", C.c_int32), ("act_scale_log2", C.c_int32)]


OUT_FIELDS = ("rgb", "depth", "depth_raw", "acc", "disp", "weights", "mask_weights", "t_vals",
              "coarse_rgb", "coarse_acc", "coarse_disp", "coarse_weights")


class NmRenderOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in OUT_FIELDS]


PREC_EXACT, PREC_FAST, PREC_FP32 = 0, 1, 2
FLAG_TRAINING, FLAG_BUFF, FLAG_TEACHER_T, FLAG_RANDOM_VOXELS = 1, 2, 4, 8
NET_COARSE, NET_FINE = 0, 1

_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_int64, C.c_float
_SIGNATURES = {
    "nm_version": (C.c_int, []),
    "nm_last_error": (C.c_char_p, []),
    "nm_device_check": (C.c_int, [_I]),
    "nm_create": (C.c_int, [_I, C.POINTER(NmNetDesc), C.POINTER(NmNetDesc), C.POINTER(NmRenderCfg), C.POINTER(_P)]),
    "nm_destroy": (C.c_int, [_P]),
    "nm_set_render_cfg": (C.c_int, [_P, C.POINTER(NmRenderCfg)]),
    "nm_load_weights": (C.c_int, [_P, _I, _I, C.POINTER(C.c_char_p), C.POINTER(_P), C.POINTER(C.c_int64)]),
    "nm_load_weights_dev": (C.c_int, [_P, _I, _I, C.POINTER(C.c_char_p), C.POINTER(_P), C.POINTER(C.c_int64), _P]),
    "nm_set_tables": (C.c_int, [_P, _P, _P]),
    "nm_set_tree": (C.c_int, [_P, _P, C.c_int32]),
    "nm_point_mlp": (C.c_int, [_P, _I, _P, _P, _L, _P, _I, _P]),
    "nm_render_rays": (C.c_int, [_P, _P, _I, _P, _L, _P, _P, _P, _I, C.c_uint64, C.POINTER(NmRenderOut), _P]),
    "nm_render_image": (C.c_int, [_P, _P, _I, _I, _F, _I, _I, _I, _P, _I, C.c_uint64, C.POINTER(NmRenderOut), _P]),
    "nm_ray_bundle": (C.c_int, [_P, _P, _I, _I, _F, _I, _F, _I, _I, _P, _P, _P]),
    "nm_grid_sigma": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "nm_volume_stats": (C.c_int, [_P, _P, _L, _P]),
    "nm_marching_cubes_count": (C.c_int, [_P, _P, _I, _I, _I, _F, _P, _P]),
    "nm_marching_cubes_emit": (C.c_int, [_P, _P, _I, _I, _I, _F, _F, _P, _P, _P, _P]),
    "nm_volume_stats_dev": (C.c_int, [_P, _P, _L, _I, _P, _P, _P]),
    "nm_mc_count": (C.c_int, [_P, _P, _I, _I, _I, _F, _I, _I, _I, _I, _P, _P]),
    "nm_mc_emit": (C.c_int, [_P, _P, _I, _I, _I, _F, _I, _I, _I, _I, _L, _P, _P, _P, _P]),
    "nm_export_obj": (C.c_int, [C.c_char_p, _P, _L, _P, _L, _P, _L, _P, _L]),
    "nm_nearest": (C.c_int, [_P, _P, _L, _P, _L, _P, _P, _P]),
    "nm_mesh_sample": (C.c_int, [_P, _P, _L, _P, _L, _L, C.c_uint64, _P, _P, _P, _P]),
    "nm_query_host": (C.c_int, [_P, _P, _I, _P, _L, _P, _I, C.c_uint64, C.POINTER(NmRenderOut)]),
    "nm_render_image_host": (C.c_int, [_P, _P, _I, _I, _F, _I, _I, _I, _P, _I, C.c_uint64, C.POINTER(NmRenderOut)]),
    "nm_point_mlp_host": (C.c_int, [_P, _I, _P, _P, _L, _P, _I]),
    "nm_zero_grad": (C.c_int, [_P, _P]),
    "nm_backward_rays": (C.c_int, [_P, _P, _I, _P, _L, _P, _P, _P, _I, C.c_uint64, _P, _P, _P]),
    "nm_loss_backward": (C.c_int, [_P, _P, _I, _P, _L, _P, _P, _P, _I, C.c_uint64, _P, _P, _P]),
    "nm_get_grad": (C.c_int, [_P, _I, C.c_char_p, _P, _L, _P]),
    "nm_ray_voxel_indices": (C.c_int, [_P, _P, _I, _P, _L, _P, _P, _P, _P]),
    "nm_ray_voxel_indices_ex": (C.c_int, [_P, _P, _I, _P, _L, _P, _I, C.c_uint64, _P, _P, _P]),
    "nm_tree_integrate": (C.c_int, [_P, _P, _P, _P, _L, _P, C.c_int32, C.c_int32, _P]),
    "nm_debug_gemm": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "nm_debug_pack": (C.c_int, [C.POINTER(NmNetDesc), _I, C.POINTER(C.c_char_p), C.POINTER(_P), C.POINTER(C.c_int64), _I, _P,
                               C.c_size_t, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nm_kernel_flags": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "nm_check_flags": (C.c_int, [_P, _P]),
    "nm_ndc_rays": (C.c_int, [_P, _I, _I, _F, _F, _P, _I, _P, _L, _P, _P, _P]),
    "nm_launch_count": (C.c_int64, [_P]),
    "nm_debug_tile_schedule": (C.c_int, [_I, _L, _I, _I, _P, _L, _P]),
    "nm_set_timing": (C.c_int, [_P, _I]),
    "nm_mlp_time_ms": (C.c_double, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
}

_lib = None


class NmError(RuntimeError):
    pass


def load():
    """dlopen the library (once) and declare every entry point of include/nerfmeshes_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NmError(f"{LIB_PATH} is missing: build it with `python -m nerfmeshes_b200.build` "
                      "(there is no fallback implementation)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(rc):
    if rc != 0:
        raise NmError(load().nm_last_error().decode("utf-8", "replace") or f"nerfmeshes_b200 error {rc}")
