"""ctypes loader for the C-ABI library (bitnetmcu_b200/libbitnetmcu_b200.so, built in-tree by csrc/Makefile).

There is no Python or CPU implementation behind this module: if the CUDA library is missing the import of
anything that computes fails loudly."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BNM_LIB_PATH") or os.path.join(HERE, "libbitnetmcu_b200.so")   # override: tuning builds only

# every symbol include/bitnetmcu_b200.h declares (checked by tests/test_capi_symbols.py)
EXPORTED = [
    "ReLUNorm", "processfclayer", "processconv33ReLU", "processmaxpool22",
    "bnm_version", "bnm_last_error", "bnm_device_count",
    "bnm_model_create", "bnm_model_load_blob", "bnm_model_destroy", "bnm_model_n_classes", "bnm_model_img_bytes",
    "bnm_model_set_option", "bnm_model_get_option", "bnm_model_active_path",
    "bnm_infer_batch", "bnm_infer_batch_device", "bnm_infer_launch_count", "bnm_host_alloc", "bnm_host_free",
    "bnm_processfclayer_batch", "bnm_relunorm_batch", "bnm_conv33relu_batch", "bnm_maxpool22_batch",
    "bnm_quantize_images", "bnm_quantize_images_device",
    "bnm_infer_batch_device_gather", "bnm_device_alloc", "bnm_device_free", "bnm_ipc_export", "bnm_ipc_open", "bnm_ipc_close",
    "bnm_enable_peer_access", "bnm_emulate_inference_quantized", "bnm_infer_batch_device_f32",
    "bnm_model_n_taps", "bnm_model_tap_width", "bnm_model_tap_stride", "bnm_infer_batch_device_taps", "bnm_infer_batch_taps",
]

PATH_AUTO, PATH_LAYERS, PATH_TCGEN05 = 0, 1, 2
OPT_PATH, OPT_NF4_EXTENSION, OPT_CHUNK_IMAGES, OPT_LAUNCH_OVERLAP, OPT_CNN_FRONTEND = 1, 2, 3, 4, 5
CNN_AUTO, CNN_CUDA_CORES, CNN_TENSOR_CORES = 0, 1, 2


class BnmLayer(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("bitperweight", C.c_int32), ("n_in", C.c_uint32), ("n_out", C.c_uint32),
                ("in_channels", C.c_uint32), ("groups", C.c_uint32), ("weights", C.c_void_p), ("weight_bytes", C.c_size_t)]


MAX_GATHER_DST = 8


class BnmGather(C.Structure):
    """bnm_gather (include/bitnetmcu_b200.h): destinations of the fused result exchange."""
    _fields_ = [("n_labels_dst", C.c_uint32), ("n_logits_dst", C.c_uint32), ("labels_dst", C.c_void_p * MAX_GATHER_DST),
                ("logits_dst", C.c_void_p * MAX_GATHER_DST), ("row_offset", C.c_size_t), ("labels_u8", C.c_uint32), ("reserved", C.c_uint32)]


MAX_TAPS = 8


class BnmTaps(C.Structure):
    """bnm_taps (include/bitnetmcu_b200.h): per tap an int8 [n][stride] buffer, or NULL when the tap is not wanted."""
    _fields_ = [("act", C.c_void_p * MAX_TAPS)]


_lib = None


def load() -> C.CDLL:
    """Load the library (once).  Raises if it has not been built: the product path has no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not built -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a).  bitnetmcu_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, u32, i32, sz, i64 = C.c_void_p, C.c_uint32, C.c_int32, C.c_size_t, C.c_int64
    sig = {
        "bnm_version": (C.c_int, []), "bnm_last_error": (C.c_char_p, []), "bnm_device_count": (C.c_int, []),
        "bnm_model_create": (C.c_int, [C.c_int, C.POINTER(BnmLayer), u32, u32, C.c_int, C.POINTER(vp)]),
        "bnm_model_load_blob": (C.c_int, [vp, sz, C.c_int, C.POINTER(vp)]),
        "bnm_model_destroy": (None, [vp]),
        "bnm_model_n_classes": (u32, [vp]), "bnm_model_img_bytes": (u32, [vp]),
        "bnm_model_set_option": (C.c_int, [vp, C.c_int, i64]), "bnm_model_get_option": (i64, [vp, C.c_int]),
        "bnm_model_active_path": (C.c_int, [vp]),
        "bnm_infer_batch": (C.c_int, [vp, vp, sz, vp, vp]),
        "bnm_infer_batch_device": (C.c_int, [vp, vp, sz, vp, vp, vp]),
        "bnm_infer_launch_count": (C.c_int, [vp, sz]),
        "bnm_host_alloc": (vp, [sz]), "bnm_host_free": (None, [vp]),
        "bnm_processfclayer_batch": (C.c_int, [vp, vp, i32, u32, u32, vp, sz, C.c_int]),
        "bnm_relunorm_batch": (C.c_int, [vp, vp, vp, u32, sz]),
        "bnm_conv33relu_batch": (C.c_int, [vp, vp, u32, u32, u32, vp, sz]),
        "bnm_maxpool22_batch": (C.c_int, [vp, u32, vp, sz]),
        "bnm_quantize_images": (C.c_int, [vp, sz, u32, vp]),
        "bnm_quantize_images_device": (C.c_int, [vp, sz, u32, vp, vp]),
        "bnm_infer_batch_device_gather": (C.c_int, [vp, vp, sz, vp, vp, C.POINTER(BnmGather), vp]),
        "bnm_device_alloc": (C.c_int, [C.c_int, sz, C.POINTER(vp)]), "bnm_device_free": (None, [vp]),
        "bnm_ipc_export": (C.c_int, [vp, vp]), "bnm_ipc_open": (C.c_int, [C.c_int, vp, C.POINTER(vp)]), "bnm_ipc_close": (C.c_int, [vp]),
        "bnm_enable_peer_access": (C.c_int, [C.c_int, C.c_int]),
        "bnm_emulate_inference_quantized": (C.c_int, [vp, vp, sz, vp]),
        "bnm_infer_batch_device_f32": (C.c_int, [vp, vp, sz, vp, vp, vp]),
        "bnm_model_n_taps": (u32, [vp]), "bnm_model_tap_width": (u32, [vp, u32]), "bnm_model_tap_stride": (u32, [vp, u32]),
        "bnm_infer_batch_device_taps": (C.c_int, [vp, vp, sz, vp, vp, C.POINTER(BnmTaps), vp]),
        "bnm_infer_batch_taps": (C.c_int, [vp, vp, sz, vp, vp, C.POINTER(BnmTaps)]),
        "ReLUNorm": (u32, [vp, vp, u32]),
        "processfclayer": (None, [vp, vp, i32, u32, u32, vp]),
        "processconv33ReLU": (vp, [vp, vp, u32, u32, vp]),
        "processmaxpool22": (vp, [vp, u32, vp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    _lib = lib
    return lib


class BnmError(RuntimeError):
    pass


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise BnmError(f"{what} failed (rc={rc}): {load().bnm_last_error().decode(errors='replace')}")
