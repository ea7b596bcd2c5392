"""ctypes binding of libdorpatch.so (the C ABI declared in include/dorpatch.h).

There is no CPU fallback: if the shared library is missing or cannot be loaded this module
raises, and every caller on the product path fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libdorpatch.so")
ABI_VERSION = 7

c_i32, c_i64, c_f32, c_vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p


class DpConfig(C.Structure):
    _fields_ = [("device", c_i32), ("img", c_i32), ("n_classes", c_i32), ("precision", c_i32),
                ("chunk", c_i32), ("max_images", c_i32), ("autotune", c_i32), ("reserved", c_i32)]


class DpAttackArgs(C.Structure):
    _fields_ = [("B", c_i32), ("S", c_i32), ("S_total", c_i32), ("stage", c_i32),
                ("x", c_vp), ("mask", c_vp), ("pattern", c_vp),
                ("rects_host", c_vp), ("y_host", c_vp), ("targeted_host", c_vp),
                ("confidence", c_f32), ("eps", c_f32),
                ("grad_adv", c_vp), ("loss_adv_host", c_vp), ("preds_host", c_vp),
                ("loss_struc_host", c_vp), ("loss_density_host", c_vp), ("group_lasso_host", c_vp),
                ("l2_host", c_vp), ("xform_host", c_vp)]


class DpUpdateArgs(C.Structure):
    _fields_ = [("B", c_i32), ("stage", c_i32),
                ("x", c_vp), ("mask", c_vp), ("pattern", c_vp), ("grad_adv", c_vp),
                ("lr_host", c_vp), ("structured_host", c_vp), ("coeff_gl_host", c_vp),
                ("density", c_f32), ("clip_min", c_f32), ("clip_max", c_f32),
                ("grad_pattern_out", c_vp), ("grad_mask_out", c_vp), ("grad_pattern_bias", c_vp)]


# name -> (restype, argtypes); every symbol include/dorpatch.h declares
SIGNATURES = {
    "dp_abi_version": (c_i32, []),
    "dp_last_error": (C.c_char_p, []),
    "dp_engine_create": (c_i32, [C.POINTER(DpConfig), C.POINTER(c_vp)]),
    "dp_engine_destroy": (None, [c_vp]),
    "dp_engine_load_weights": (c_i32, [c_vp, c_i32, C.POINTER(C.c_char_p), C.POINTER(c_vp), C.POINTER(c_i64)]),
    "dp_engine_device_bytes": (c_i64, [c_vp]),
    "dp_engine_launch_count": (c_i64, [c_vp]),
    "dp_engine_graph_replays": (c_i64, [c_vp]),
    "dp_engine_graph_status": (C.c_char_p, [c_vp]),
    "dp_engine_profile": (c_i32, [c_vp, c_i32]),
    "dp_engine_profile_read": (c_i32, [c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, C.POINTER(c_i32)]),
    "dp_paste": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_f32, c_vp, c_vp, c_vp, c_vp]),
    "dp_window_sum": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "dp_expand": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "dp_expand_dev": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "dp_debug_k1_tuning": (c_i32, [c_i32, c_i32, c_i32]),
    "dp_debug_k1_last": (c_i32, [c_vp]),
    "dp_k1_samples_per_launch": (c_i32, [c_vp, c_i32]),
    "dp_expand_step_dev": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp]),
    "dp_input_layout": (c_i32, [c_vp, C.POINTER(c_i32), C.POINTER(c_i32)]),
    "dp_predict": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "dp_attack_grad": (c_i32, [c_vp, C.POINTER(DpAttackArgs), c_vp]),
    "dp_attack_update": (c_i32, [c_vp, C.POINTER(DpUpdateArgs), c_vp]),
    "dp_attack_step_host": (c_i32, [c_vp, C.POINTER(DpAttackArgs), C.POINTER(DpUpdateArgs), c_vp]),
    "dp_net_forward_backward": (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "dp_failed_set_write": (c_i32, [c_vp, c_i32, c_vp, c_i32, c_vp]),
    "dp_failed_set_update": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_f32, c_vp, c_vp]),
    "dp_failed_set_read": (c_i32, [c_vp, c_i32, c_vp, c_i32, c_vp, c_vp]),
    "dp_debug_k1t": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "dp_debug_cw": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_f32, c_f32, c_vp, c_vp, c_vp, c_i32, c_i32, c_vp]),
    "dp_debug_gn_gemm": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "dp_debug_gn": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
}

_lib = None


def load():
    """dlopen libdorpatch.so (RTLD_GLOBAL not needed) and type every entry point."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libdorpatch.so is not built (%s). Run `python -m dorpatch_b200.build` "
            "(or __graft_entry__.build()). There is no CPU fallback." % LIB_PATH)
    import torch  # noqa: F401  -- loads the CUDA runtime / cuDNN / cuBLAS copies the library binds to
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    v = lib.dp_abi_version()
    if v != ABI_VERSION:
        raise RuntimeError("libdorpatch.so ABI version %d != expected %d; rebuild" % (v, ABI_VERSION))
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError("libdorpatch: " + load().dp_last_error().decode("utf-8", "replace"))
