"""CPU checks of the untangling entry points: hdgnn_hunk_groups and hdgnn_set_predictions reject bad arguments before any
CUDA call, so they need no GPU."""
import ctypes as C

import torch


def test_hunk_groups_validates_arguments_without_a_gpu():
    from hdgnn_b200 import _lib
    f = _lib.lib.hdgnn_hunk_groups
    bits, groups, ngroups = C.c_void_p(0x10000), C.c_void_p(0x20000), C.c_void_p(0x30000)      # never dereferenced
    bad = [
        (1, 1, bits, groups, ngroups),                      # n below 2
        (1, 513, bits, groups, ngroups),                    # n above HDGNN_MAX_N
        (0, 74, bits, groups, ngroups),                     # B below 1
        (1, 74, None, groups, ngroups),                     # null bits
        (1, 74, bits, None, ngroups),                       # null groups
        (1, 74, C.c_void_p(0x10004), groups, ngroups),      # bits not 16-byte aligned
        (1, 74, bits, C.c_void_p(0x20002), ngroups),        # groups not 4-byte aligned
        (1, 74, bits, groups, C.c_void_p(0x30001)),         # ngroups not 4-byte aligned
    ]
    for B, n, b, g, ng in bad:
        assert f(B, n, b, g, ng, None) == _lib.E_INVALID, (B, n, b, g, ng)
    if not torch.cuda.is_available():                        # valid arguments reach the device and fail loudly there
        assert f(1, 74, bits, groups, None, None) == _lib.E_CUDA


def test_set_predictions_validates_arguments_without_a_gpu():
    from hdgnn_b200 import _lib
    assert _lib.lib.hdgnn_set_predictions(None, None) == _lib.E_INVALID
    assert _lib.lib.hdgnn_infer_host(None, 1, None, None, None, None, None, None, None, None, None) == _lib.E_INVALID
