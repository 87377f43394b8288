"""ctypes binding of libhdgnn.so (include/hdgnn.h).  There is no fallback: if the library is
missing or fails to load, importing this module raises."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB

OK, E_INVALID, E_CUDA, E_NOMEM, E_UNSUPPORTED, E_PEER = 0, -1, -2, -3, -4, -5
MAX_N = 512


class Config(C.Structure):
    _fields_ = [("Ne", C.c_int32), ("Nc", C.c_int32), ("variant", C.c_int32), ("max_batch", C.c_int32),
                ("device", C.c_int32), ("rows_per_cta_e", C.c_int32), ("rows_per_cta_c", C.c_int32),
                ("flags", C.c_int32)]


class HdgnnError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libhdgnn error {code}: {msg}")
        self.code = code


def _load():
    if not os.path.exists(LIB):
        raise ImportError(
            f"{LIB} is missing: build it with `python -m hdgnn_b200.build` (nvcc, sm_100a). "
            "hdgnn_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB)
    vp, i32, f32 = C.c_void_p, C.c_int, C.c_float
    sig = {
        "hdgnn_param_count": ([i32], i32),
        "hdgnn_param_offset": ([i32, C.c_char_p], i32),
        "hdgnn_create": ([C.POINTER(Config), C.POINTER(vp)], i32),
        "hdgnn_destroy": ([vp], i32),
        "hdgnn_last_error": ([vp], C.c_char_p),
        "hdgnn_label_pitch": ([i32], i32),
        "hdgnn_bit_words": ([i32], i32),
        "hdgnn_forward": ([vp, i32, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp], i32),
        "hdgnn_forward_backward": ([vp, i32, i32, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp], i32),
        "hdgnn_adam_step": ([vp, vp, vp, vp, vp, vp, f32, f32, f32, f32, vp, vp], i32),
        "hdgnn_train_step": ([vp, i32, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, f32, f32, f32, f32, vp, vp, vp, vp], i32),
        "hdgnn_train_step_host": ([vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, f32, f32, f32, f32, vp, vp, vp], i32),
        "hdgnn_forward_backward_host": ([vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp], i32),
        "hdgnn_peer_export": ([vp, i32, vp], i32),
        "hdgnn_peer_attach": ([vp, i32, i32, vp], i32),
        "hdgnn_peer_status": ([vp], i32),
        "hdgnn_set_hits_accumulator": ([vp, vp], i32),
        "hdgnn_set_eval_counters": ([vp, vp], i32),
        "hdgnn_set_predictions": ([vp, vp], i32),
        "hdgnn_train_step_peer": ([vp, i32, i32, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, f32, f32, f32, f32, vp, vp, vp, vp], i32),
        "hdgnn_train_step_peer_host": ([vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, f32, f32, f32, f32, vp, vp, vp], i32),
        "hdgnn_infer_host": ([vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp], i32),
        "hdgnn_normalize_propagate": ([i32, i32, vp, i32, vp, i32, vp, vp, i32, f32, i32, vp, vp, vp], i32),
        "hdgnn_map_conv": ([i32, i32, vp, i32, vp, vp, f32, f32, i32, vp, vp, vp], i32),
        "hdgnn_propagate_backward_work": ([i32, i32, i32, i32], C.c_size_t),
        "hdgnn_normalize_propagate_backward": ([i32, i32, vp, i32, vp, i32, vp, i32, f32, i32, vp, vp, vp, vp, vp, vp, vp], i32),
        "hdgnn_map_conv_backward": ([i32, i32, vp, i32, vp, vp, f32, f32, i32, f32, vp, vp, vp, vp], i32),
        "hdgnn_compact_from_raw": ([i32, i32, vp, i32, vp, i32, vp, vp, vp], i32),
        "hdgnn_pack_label_bits": ([i32, i32, vp, i32, vp, vp], i32),
        "hdgnn_eval_counts": ([i32, i32, vp, vp, i32, vp, vp, i32, vp], i32),
        "hdgnn_hunk_groups": ([i32, i32, vp, vp, vp, vp], i32),
        "hdgnn_partition_counts": ([i32, i32, vp, vp, vp, vp, vp], i32),
        "hdgnn_hunk_clusters_work": ([i32, i32], C.c_size_t),
        "hdgnn_hunk_clusters": ([i32, i32, vp, vp, f32, vp, vp, vp, vp], i32),
        "hdgnn_hunk_linkage": ([i32, i32, vp, vp, vp, vp, vp, vp, vp], i32),
        "hdgnn_linkage_cut": ([i32, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp], i32),
        "hdgnn_workspace": ([vp, C.c_char_p, C.POINTER(vp), C.POINTER(C.c_size_t)], i32),
        "hdgnn_workspace_copy": ([vp, C.c_char_p, vp, C.c_size_t, vp], i32),
        "hdgnn_profile": ([vp, i32], i32),
        "hdgnn_profile_count": ([vp], i32),
        "hdgnn_profile_get": ([vp, i32, C.c_char_p, i32, C.POINTER(f32)], i32),
        "hdgnn_last_launch_count": ([vp], i32),
        "hdgnn_measure_fp32_peak": ([i32, C.POINTER(f32)], i32),
    }
    for name, (argtypes, restype) in sig.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.argtypes = argtypes
        fn.restype = restype
    return lib, sorted(sig)


lib, EXPORTS = _load()


def check(rc: int, handle=None):
    if rc != OK:
        msg = lib.hdgnn_last_error(handle)
        raise HdgnnError(rc, msg.decode() if msg else "")
