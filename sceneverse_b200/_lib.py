"""ctypes binding of libsvpointops (include/svpointops.h).  No fallback: if the CUDA library is
missing or a call fails this raises — the product path never routes around the native code."""
import ctypes
import os

_LIBDIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib")
_cache = {}

c_int, c_float, c_void_p = ctypes.c_int, ctypes.c_float, ctypes.c_void_p

_POINTOPS_SIGS = {
    # name: argtypes
    "sv_fps_f32": [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "sv_gather_points_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_gather_points_grad_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_ball_query_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p],
    "sv_group_points_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_group_points_grad_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_three_nn_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "sv_three_interpolate_f32": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_three_interpolate_grad_f32": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_fps_ballquery_f32": [c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "sv_scene_prep_f32": [c_void_p, c_void_p, c_int, c_int, ctypes.c_ulonglong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "sv_token_mask": [c_void_p, c_void_p, ctypes.c_longlong, c_float, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_ulonglong,
                      c_void_p, c_void_p, c_void_p],
    "sv_coin_mask": [c_void_p, ctypes.c_longlong, c_float, ctypes.c_ulonglong, c_void_p, c_void_p],
    "sv_sa_sample_f32": [c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p, c_void_p,
                         c_int, c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
}


class NativeLibraryError(RuntimeError):
    pass


def _load(name):
    if name in _cache:
        return _cache[name]
    path = os.path.join(_LIBDIR, name)
    if not os.path.exists(path):
        raise NativeLibraryError(
            f"{path} is missing: build it with `python -m sceneverse_b200.build` "
            "(sceneverse_b200 has no CPU or PyTorch fallback)")
    lib = ctypes.CDLL(path)
    _cache[name] = lib
    return lib


def pointops():
    lib = _load("libsvpointops.so")
    if not getattr(lib, "_sv_ready", False):
        for fn, argtypes in _POINTOPS_SIGS.items():
            f = getattr(lib, fn)
            f.argtypes = argtypes
            f.restype = c_int
        lib.sv_version.restype = c_int
        lib.sv_status_string.restype = ctypes.c_char_p
        lib.sv_status_string.argtypes = [c_int]
        lib.sv_last_cuda_error.restype = c_int
        lib.sv_last_cuda_error_string.restype = ctypes.c_char_p
        lib.sv_launch_count.restype = ctypes.c_ulonglong
        lib._sv_ready = True
    return lib


_GPS_SIGS = {
    "sv_tc05_selftest": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    "sv_gemm_bf16": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int,
                     c_int, c_int, c_void_p],
    "sv_gemm_bf16_ex": [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p,
                        c_void_p, c_int, c_int, c_int, c_void_p],
    "sv_attention_fwd_bf16": [c_void_p, ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p,
                              ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_int,
                              c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p],
    "sv_pairwise_locs_f32": [c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p],
    "sv_cross_entropy_fwd_bwd": [c_void_p, ctypes.c_longlong, c_int, c_void_p, c_int, c_int, ctypes.c_longlong, c_void_p,
                                 c_void_p, c_void_p],
    "sv_cross_entropy_fwd_bwd_strided": [c_void_p, ctypes.c_longlong, c_int, c_void_p, c_int, c_int, ctypes.c_longlong,
                                         c_void_p, c_void_p, ctypes.c_longlong, c_void_p],
    "sv_normalize_allgather_f32": [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                   ctypes.c_uint, c_void_p],
    "sv_normalize_allgather_dev_f32": [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                       c_void_p, c_void_p],
    "sv_attention_fwd_lse_bf16": [c_void_p, ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p,
                                  ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_int,
                                  c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p],
    "sv_attention_bwd_bf16": [c_void_p, ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p,
                              ctypes.c_longlong, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                              c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "sv_attention_fwd_dropout_bf16": [c_void_p, ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p,
                                      ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p,
                                      c_int, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_float,
                                      ctypes.c_ulonglong, c_void_p],
    "sv_attention_bwd_dropout_bf16": [c_void_p, ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p,
                                      ctypes.c_longlong, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_float, ctypes.c_ulonglong, c_void_p],
    "sv_attention_bwd_strided_bf16": [c_void_p, ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p,
                                      ctypes.c_longlong, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                      c_void_p, c_float, ctypes.c_ulonglong, c_void_p],
    "sv_attention_bwd_scratch_floats": [c_int, c_int, c_int, c_int],
    "sv_layer_norm_fwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_float, ctypes.c_ulonglong,
                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "sv_layer_norm_bwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_float, ctypes.c_ulonglong,
                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "sv_layer_norm_bwd_acc": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_float, ctypes.c_ulonglong,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p],
    "sv_layer_norm_scratch_floats": [c_int],
    "sv_dropout_seed_offset": [c_void_p],
    "sv_colsum": [c_void_p, ctypes.c_longlong, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "sv_colsum_scratch_floats": [c_int],
    "sv_l2norm_fwd": [c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p],
    "sv_l2norm_bwd": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p],
    "sv_gemm_force_ctas": [c_int],
    "sv_gemm_profile": [c_void_p],
    "sv_mma_bench": [c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_linear_fwd_bf16": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_float, ctypes.c_ulonglong,
                           c_void_p, c_int, c_int, c_void_p, c_void_p],
    "sv_linear_dgrad_bf16": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_float,
                             ctypes.c_ulonglong, c_void_p, c_int, c_int, c_void_p],
    "sv_linear_wgrad_bf16": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p],
    "sv_act_bwd_bf16": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p],
    "sv_embedding_bwd": [c_void_p, ctypes.c_longlong, c_int, c_void_p, c_int, c_int, ctypes.c_longlong, ctypes.c_longlong,
                         c_void_p, c_void_p],
    "sv_scale_inplace": [c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p],
    "sv_adamw_scratch_floats": [],
    "sv_adamw_flat": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_longlong, c_void_p, c_int, c_float, c_void_p,
                      c_void_p, c_float, c_float, c_float, c_float, c_void_p, c_void_p, c_void_p],
    "sv_pn_group_rows": [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_pn_group_rows_grad": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_pn_scratch_floats": [c_int],
    "sv_pn_bn_relu_fwd": [c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                          c_void_p, c_void_p],
    "sv_pn_bn_relu_bwd": [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                          c_void_p, c_int, c_void_p, c_void_p],
    "sv_pn_rowgroup_max": [c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "sv_pn_rowgroup_max_grad": [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p, c_void_p],
    "sv_sa_mlp_param_bytes": [c_int],
    "sv_sa1_mlp_bf16": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "sv_sa2_mlp_bf16": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
}


def gps():
    lib = _load("libsvgps.so")
    if not getattr(lib, "_sv_ready", False):
        for fn, argtypes in _GPS_SIGS.items():
            f = getattr(lib, fn)
            f.argtypes = argtypes
            f.restype = c_int
        lib.svgps_launch_count.restype = ctypes.c_ulonglong
        lib.svgps_last_cuda_error_string.restype = ctypes.c_char_p
        # status strings live in libsvpointops
        lib.sv_status_string = pointops().sv_status_string
        lib.sv_last_cuda_error_string = lib.svgps_last_cuda_error_string
        lib._sv_ready = True
    return lib


def check(lib, status, what):
    if status != 0:
        msg = lib.sv_status_string(status).decode()
        if status == 2:
            msg += ": " + lib.sv_last_cuda_error_string().decode()
        raise RuntimeError(f"{what} failed: {msg}")


def launch_count():
    """Kernel launches enqueued so far by both native libraries."""
    n = int(pointops().sv_launch_count())
    import os as _os
    if _os.path.exists(_os.path.join(_LIBDIR, "libsvgps.so")):
        n += int(gps().svgps_launch_count())
    return n
