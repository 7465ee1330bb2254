"""ctypes binding of libcld_b200.so (C ABI in include/cld_b200.h).

The library is built in-tree by `__graft_entry__.build()` / `csrc/Makefile`.  There is no CPU or
PyTorch fallback: if the shared object is missing, importing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CLD_B200_LIB") or os.path.join(_HERE, "libcld_b200.so")   # override: A/B of two builds

CLD_PREC_FP32, CLD_PREC_BF16 = 0, 1
CLD_SAMPLER_DDPM, CLD_SAMPLER_DDIM = 0, 1
CLD_OPT_ADAM, CLD_OPT_SGD = 0, 1

EXPORTS = [
    "cld_version", "cld_create", "cld_destroy", "cld_last_error", "cld_load_unet", "cld_load_decoder",
    "cld_set_schedule", "cld_unet_forward", "cld_unet_debug_stage", "cld_posterior_step", "cld_add_noise",
    "cld_decode_rollout", "cld_unicycle", "cld_indicators", "cld_guidance_step", "cld_sample",
    "cld_launch_count", "cld_profile_begin", "cld_profile_end", "cld_tc_selftest",
    "cld_unet_train_forward", "cld_unet_backward", "cld_ppo_head", "cld_mse_head", "cld_ppo_grad", "cld_adam_step", "cld_adam_step_dev", "cld_train_set_precision",
    "cld_context_create", "cld_context_destroy", "cld_context_last_error", "cld_context_load", "cld_context_forward", "cld_context_forward_history",
    "cld_context_launch_count", "cld_context_conv_flops",
]


class CldConfig(C.Structure):
    _fields_ = [
        ("horizon", C.c_int32), ("latent_dim", C.c_int32), ("cond_dim", C.c_int32), ("base_dim", C.c_int32),
        ("dims", C.c_int32 * 3), ("hidden", C.c_int32), ("n_timesteps", C.c_int32), ("max_rows", C.c_int32),
        ("precision", C.c_int32), ("dt", C.c_float), ("acce_lo", C.c_float), ("acce_hi", C.c_float),
        ("v_lo", C.c_float), ("v_hi", C.c_float), ("max_steer", C.c_float), ("max_yawvel", C.c_float),
        ("norm_mean", C.c_float * 6), ("norm_std", C.c_float * 6),
    ]


class CldGuidanceConfig(C.Structure):
    _fields_ = [
        ("w_agent_collision", C.c_float), ("w_map_collision", C.c_float), ("w_target_pos", C.c_float),
        ("num_disks", C.c_int32), ("buffer_dist", C.c_float), ("decay_rate", C.c_float),
        ("num_points_l", C.c_int32), ("num_points_w", C.c_int32), ("speed_th", C.c_float),
        ("min_target_time", C.c_float), ("optimizer", C.c_int32), ("lr", C.c_float),
        ("w_target_speed", C.c_float), ("w_acc_limit", C.c_float), ("acc_limit", C.c_float),
        ("w_speed_limit", C.c_float), ("speed_limit", C.c_float), ("w_waypoint", C.c_float),
        ("grad_steps", C.c_int32),
    ]


class CldScene(C.Structure):
    _fields_ = [
        ("num_scenes", C.c_int32), ("agents_per_scene", C.c_int32), ("num_samp", C.c_int32),
        ("extent", C.c_void_p), ("world_from_agent", C.c_void_p), ("raster_from_agent", C.c_void_p),
        ("curr_speed", C.c_void_p), ("drivable_map", C.c_void_p), ("map_h", C.c_int32), ("map_w", C.c_int32),
        ("target_pos", C.c_void_p), ("others_pos", C.c_void_p), ("others_avail", C.c_void_p),
        ("num_others", C.c_int32), ("map_packed", C.c_int32), ("target_speed", C.c_void_p),
        ("wp_target", C.c_void_p), ("wp_mode", C.c_void_p), ("wp_time", C.c_void_p), ("wp_dist", C.c_void_p), ("wp_weight", C.c_void_p),
        ("scene_start", C.c_void_p), ("scene_start_host", C.c_void_p),
    ]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libcld_b200.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C %s/csrc`.  cld_b200 has no CPU / PyTorch fallback." % (LIB_PATH, _HERE))
    lib = C.CDLL(LIB_PATH)
    vp, i32, u64 = C.c_void_p, C.c_int, C.c_uint64
    lib.cld_version.restype = C.c_int
    lib.cld_create.argtypes = [C.POINTER(CldConfig), C.POINTER(vp)]
    lib.cld_destroy.argtypes = [vp]
    lib.cld_destroy.restype = None
    lib.cld_last_error.argtypes = [vp]
    lib.cld_last_error.restype = C.c_char_p
    lib.cld_load_unet.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_int64), i32, vp]
    lib.cld_load_decoder.argtypes = [vp, C.POINTER(vp), i32, vp]
    lib.cld_set_schedule.argtypes = [vp] + [C.POINTER(C.c_float)] * 7 + [i32]
    lib.cld_unet_forward.argtypes = [vp, vp, vp, vp, vp, i32, vp]
    f32 = C.c_float
    lib.cld_unet_train_forward.argtypes = [vp, vp, vp, vp, vp, i32, vp]
    lib.cld_unet_backward.argtypes = [vp, vp, C.POINTER(vp), i32, vp, i32, vp]
    lib.cld_ppo_head.argtypes = [vp, vp, vp, vp, vp, vp, vp, f32, vp, f32, vp, vp, vp, i32, vp]
    lib.cld_mse_head.argtypes = [vp, vp, vp, vp, vp, i32, vp]
    lib.cld_ppo_grad.argtypes = [vp, vp, vp, vp, vp, vp, vp, f32, vp, f32, C.POINTER(vp), i32, vp, vp, i32, vp]
    f64 = C.c_double
    lib.cld_adam_step.argtypes = [vp, vp, vp, vp, vp, C.c_int64, f64, f64, f64, f64, f64, i32, vp]
    lib.cld_adam_step_dev.argtypes = [vp, vp, vp, vp, vp, C.c_int64, vp, vp, f64, f64, f64, f64, vp]
    lib.cld_train_set_precision.argtypes = [vp, i32]
    lib.cld_unet_debug_stage.argtypes = [vp, i32, vp, i32, vp]
    lib.cld_posterior_step.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp, i32, vp]
    lib.cld_add_noise.argtypes = [vp, vp, vp, i32, vp, i32, vp]
    lib.cld_decode_rollout.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp]
    lib.cld_unicycle.argtypes = [vp, vp, vp, vp, i32, vp]
    lib.cld_indicators.argtypes = [vp, vp, C.POINTER(CldScene), vp, vp, vp, i32, vp]
    lib.cld_guidance_step.argtypes = [vp, vp, vp, vp, C.POINTER(CldScene), C.POINTER(CldGuidanceConfig), vp, vp, vp,
                                      i32, vp]
    lib.cld_sample.argtypes = [vp, vp, vp, u64, C.c_int64, vp, vp, C.POINTER(CldScene), C.POINTER(CldGuidanceConfig), i32, i32,
                               vp, vp, C.POINTER(C.c_int), vp, vp, vp, i32, vp]
    lib.cld_tc_selftest.argtypes = [vp, i32, vp, i32, i32, i32, i32, i32, i32, vp, vp]
    lib.cld_launch_count.argtypes = [vp]
    lib.cld_profile_begin.argtypes = [vp]
    lib.cld_profile_end.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_int), i32]
    lib.cld_context_create.argtypes = [i32, C.POINTER(vp)]
    lib.cld_context_destroy.argtypes = [vp]
    lib.cld_context_last_error.argtypes = [vp]
    lib.cld_context_load.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_int64), i32, vp]
    lib.cld_context_forward.argtypes = [vp, vp, vp, i32, vp, vp, i32, vp, vp]
    lib.cld_context_forward_history.argtypes = [vp, vp, vp, vp, vp, i32, vp, i32, vp, vp, vp, vp]
    lib.cld_context_launch_count.argtypes = [vp]
    lib.cld_context_conv_flops.argtypes = [vp]
    special = ("cld_destroy", "cld_last_error", "cld_launch_count", "cld_context_destroy", "cld_context_last_error",
               "cld_context_launch_count", "cld_context_conv_flops")
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in special:
            fn.restype = C.c_int
    lib.cld_launch_count.restype = C.c_ulonglong
    lib.cld_context_destroy.restype = None
    lib.cld_context_last_error.restype = C.c_char_p
    lib.cld_context_launch_count.restype = C.c_ulonglong
    lib.cld_context_conv_flops.restype = C.c_double
    return lib


lib = _load()
