"""ctypes binding of the C-ABI (include/nvwn_b200.h, include/wavenet_infer.h).

There is no CPU fallback and no pure-Python path: if the CUDA library is missing this raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NVWN_LIB_PATH") or os.path.join(HERE, "lib", "libwavenet_infer.so")      # (override: experimental builds)

FP32, FP16, FP32_FAST = 0, 1, 2
KERNEL_AUTO, KERNEL_STREAM, KERNEL_TENSORCORE, KERNEL_LATENCY = 0, 16, 17, 18

_vp = C.c_void_p


class LaunchInfo(C.Structure):
    _fields_ = [("kernel", C.c_int), ("grid", C.c_int), ("block", C.c_int), ("smem_bytes", C.c_int),
                ("batch_per_cta", C.c_int), ("cluster", C.c_int),
                ("launches", C.c_ulonglong), ("weight_bytes", C.c_ulonglong)]


# every symbol include/*.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "nvwn_create": (C.c_int, [C.POINTER(_vp)] + [C.c_int] * 10),
    "nvwn_create_windowed": (C.c_int, [C.POINTER(_vp)] + [C.c_int] * 10),
    "nvwn_destroy": (C.c_int, [_vp]),
    "nvwn_last_error": (C.c_char_p, []),
    "nvwn_set_embeddings": (C.c_int, [_vp, _vp, _vp]),
    "nvwn_set_layer_weights": (C.c_int, [_vp, C.c_int] + [_vp] * 7),
    "nvwn_set_out_weights": (C.c_int, [_vp] + [_vp] * 4),
    "nvwn_set_inputs": (C.c_int, [_vp, _vp, _vp]),
    "nvwn_set_selectors": (C.c_int, [_vp, _vp]),
    "nvwn_set_conditioning": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp]),
    "nvwn_set_selectors_random": (C.c_int, [_vp, C.c_ulonglong, _vp]),
    "nvwn_set_selectors_range": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp]),
    "nvwn_set_selectors_random_range": (C.c_int, [_vp, C.c_ulonglong, C.c_int, C.c_int, _vp]),
    "nvwn_libc_selectors": (C.c_int, [_vp, C.c_int, C.c_int]),
    "nvwn_reset_history": (C.c_int, [_vp]),
    "nvwn_set_forced": (C.c_int, [_vp, _vp]),
    "nvwn_weight_blob": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(C.c_ulonglong)]),
    "nvwn_weights_updated": (C.c_int, [_vp]),
    "nvwn_run_partial": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _vp]),
    "nvwn_run": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int, _vp]),
    "nvwn_get_yout": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp]),
    "nvwn_get_audio": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "nvwn_mulaw_table": (C.c_int, [C.c_int, _vp, _vp, _vp]),
    "nvwn_set_conditioning_from_features": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, _vp]),
    "nvwn_cond_producer_load": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp]),
    "nvwn_cond_producer_run": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp]),
    "nvwn_cond_from_features_host": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int]),
    "nvwn_get_xt_out": (C.c_int, [_vp, C.c_int, _vp]),
    "nvwn_get_skip_out": (C.c_int, [_vp, C.c_int, _vp]),
    "nvwn_get_zs": (C.c_int, [_vp, _vp]),
    "nvwn_get_za": (C.c_int, [_vp, _vp]),
    "nvwn_get_p": (C.c_int, [_vp, _vp]),
    "nvwn_get_launch_info": (C.c_int, [_vp, C.POINTER(LaunchInfo)]),
    "nvwn_device_count": (C.c_int, []),
    "nvwn_set_device": (C.c_int, [C.c_int]),
    "wavenet_infer_fp16": (None, [C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int] + [C.POINTER(_vp)] * 7
                           + [_vp, _vp, C.c_int, _vp, C.c_int, _vp]),
    "wavenet_infer": (None, [C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int] + [C.POINTER(_vp)] * 7
                      + [_vp, _vp, C.c_int, _vp, C.c_int, _vp]),
    "get_R": (C.c_int, []),
    "get_S": (C.c_int, []),
    "get_A": (C.c_int, []),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m nv_wavenet_b200.build` "
                "(nvcc, sm_100a).  nv_wavenet_b200 has no CPU or PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)          # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


class NvwnError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != 0:
        msg = lib().nvwn_last_error()
        raise NvwnError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
