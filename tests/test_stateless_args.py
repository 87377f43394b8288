"""Argument checks of the nine stateless entry points (no handle) and of their Python wrappers.

Every entry point refuses a bad argument before its first CUDA call, so these run without a GPU: the call returns the expected
code and hdgnn_last_error(NULL) names the entry point and the argument.  Valid arguments reach the device, and without one the
call fails loudly (HDGNN_E_CUDA).  The wrappers check the shapes the C call derives its sizes from before they check for CUDA
tensors, so wrong shapes raise ValueError on the CPU as well."""
import ctypes as C

import pytest
import torch

from hdgnn_b200 import _lib
from hdgnn_b200._lib import E_CUDA, E_INVALID, lib

NAN = float("nan")


def P(addr):
    """A fake device pointer: never dereferenced, the calls below are refused (or fail) before any launch."""
    return C.c_void_p(addr)


# entry point -> (parameter names without the stream, valid arguments, bad cases).  A case changes some arguments; the first
# one it names is the argument the message must name.  Pointers are distinct multiples of 64 KB, so each is aligned.
TABLE = {
    "hdgnn_hunk_groups": (
        "B n bits groups ngroups",
        (1, 74, P(0x10000), P(0x20000), P(0x30000)),
        [dict(n=1), dict(n=513), dict(B=0), dict(bits=None), dict(groups=None),
         dict(bits=P(0x10004)), dict(groups=P(0x20002)), dict(ngroups=P(0x30001))]),
    "hdgnn_partition_counts": (
        "B n pred truth nh counts",
        (1, 74, P(0x10000), P(0x20000), P(0x30000), P(0x40000)),
        [dict(B=0), dict(n=1), dict(n=513), dict(pred=None), dict(truth=None), dict(counts=None),
         dict(pred=P(0x10002)), dict(truth=P(0x20001)), dict(nh=P(0x30003)), dict(counts=P(0x40004))]),
    "hdgnn_hunk_clusters": (
        "B n probs nh threshold groups ngroups work",
        (1, 74, P(0x10000), P(0x20000), 0.5, P(0x30000), P(0x40000), P(0x50000)),
        [dict(n=1), dict(n=513), dict(B=0), dict(probs=None), dict(groups=None), dict(threshold=NAN),
         dict(probs=P(0x10002)), dict(nh=P(0x20001)), dict(groups=P(0x30002)), dict(ngroups=P(0x40003)),
         dict(work=P(0x50002), n=300),
         dict(work=None, n=300)]),                  # above n = 169 the tables need the workspace
    "hdgnn_compact_from_raw": (
        "N n raw raw_is_f64 grid pitch diag err",
        (2, 74, P(0x10000), 1, P(0x20000), 80, P(0x30000), P(0x40000)),
        [dict(N=0), dict(n=1), dict(n=513), dict(pitch=64), dict(pitch=88), dict(pitch=544), dict(raw=None), dict(grid=None),
         dict(N=1 << 22, n=512, pitch=512),        # more than 2^31 - 1 rows
         dict(raw=P(0x10004)), dict(raw=P(0x10002), raw_is_f64=0), dict(diag=P(0x30002)), dict(err=P(0x40001))]),
    "hdgnn_eval_counts": (
        "B Nc probs Y y_pitch counts auc auc_first",
        (2, 74, P(0x10000), P(0x20000), 80, P(0x30000), P(0x40000), 0),
        [dict(B=0), dict(Nc=1), dict(Nc=513), dict(y_pitch=73), dict(probs=None), dict(Y=None), dict(counts=None),
         dict(probs=P(0x10002)), dict(counts=P(0x30004)), dict(auc=P(0x40004))]),
    "hdgnn_pack_label_bits": (
        "N n grid pitch bits",
        (2, 74, P(0x10000), 80, P(0x20000)),
        [dict(N=0), dict(n=1), dict(n=513), dict(pitch=64), dict(pitch=88), dict(pitch=544), dict(grid=None), dict(bits=None),
         dict(grid=P(0x10008)), dict(bits=P(0x20004))]),
    "hdgnn_normalize_propagate": (
        "B N adj adj_pitch H d_in W bias d_out eps flags out dinv_out",
        (2, 74, P(0x10000), 80, P(0x20000), 20, P(0x30000), P(0x40000), 20, 1e-3, 0, P(0x50000), P(0x60000)),
        [dict(B=0), dict(N=1), dict(N=513), dict(adj=None), dict(adj=P(0x10008)), dict(adj_pitch=64), dict(adj_pitch=88),
         dict(adj_pitch=80, flags=32),             # a label bitmap's pitch is 4 * bit_words(N) = 16
         dict(d_in=0), dict(d_in=33), dict(d_out=33), dict(W=None, d_out=10), dict(H=None), dict(out=None),
         dict(H=P(0x20002)), dict(W=P(0x30002)), dict(bias=P(0x40001)), dict(out=P(0x50002)), dict(dinv_out=P(0x60003))]),
    "hdgnn_map_conv": (
        "B N adj adj_pitch x theta lam_max eps flags per_commit loss",
        (2, 74, P(0x10000), 80, P(0x20000), P(0x30000), 1.5, 1e-3, 0, P(0x40000), P(0x50000)),
        [dict(B=0), dict(N=513), dict(adj=P(0x10004)), dict(adj_pitch=32, flags=32 | 4), dict(lam_max=0.0), dict(lam_max=NAN),
         dict(x=None), dict(theta=None), dict(per_commit=None),
         dict(x=P(0x20002)), dict(theta=P(0x30001)), dict(per_commit=P(0x40002)), dict(loss=P(0x50003))]),
    "hdgnn_normalize_propagate_backward": (
        "B N adj adj_pitch H d_in W d_out eps flags out dOut dH dW dbias work",
        (2, 74, P(0x10000), 80, P(0x20000), 20, P(0x30000), 20, 1e-3, 0, P(0x40000), P(0x50000), P(0x60000), P(0x70000),
         P(0x80000), P(0x90000)),
        [dict(B=0), dict(N=513), dict(adj=None), dict(adj_pitch=72), dict(d_in=33), dict(d_out=0), dict(W=None, d_out=10),
         dict(H=None), dict(dOut=None), dict(work=None), dict(out=None, flags=2),      # P_RELU reads the forward's output
         dict(H=P(0x20002)), dict(W=P(0x30002)), dict(out=P(0x40002)), dict(dOut=P(0x50001)), dict(dH=P(0x60002)),
         dict(dW=P(0x70003)), dict(dbias=P(0x80002)), dict(work=P(0x90002))]),
    "hdgnn_map_conv_backward": (
        "B N adj adj_pitch x theta lam_max eps flags gscale dx dtheta work",
        (2, 74, P(0x10000), 80, P(0x20000), P(0x30000), 1.5, 1e-3, 0, 1.0, P(0x40000), P(0x50000), P(0x60000)),
        [dict(B=0), dict(N=1), dict(adj=None), dict(adj_pitch=80, flags=32), dict(lam_max=-1.0), dict(lam_max=NAN),
         dict(x=None), dict(theta=None), dict(work=None),                              # dtheta needs the workspace
         dict(x=P(0x20002)), dict(theta=P(0x30002)), dict(dx=P(0x40001)), dict(dtheta=P(0x50002)), dict(work=P(0x60002))]),
}


def _args(names, valid, change):
    names = names.split()
    assert set(change) <= set(names), change
    return [change.get(k, v) for k, v in zip(names, valid)]


# every optional pointer may be NULL
OPTIONAL = {"hdgnn_hunk_groups": dict(ngroups=None), "hdgnn_partition_counts": dict(nh=None),
            "hdgnn_hunk_clusters": dict(nh=None, ngroups=None, work=None), "hdgnn_compact_from_raw": dict(diag=None, err=None),
            "hdgnn_eval_counts": dict(auc=None), "hdgnn_pack_label_bits": {},
            "hdgnn_normalize_propagate": dict(W=None, bias=None, dinv_out=None),
            "hdgnn_map_conv": dict(loss=None), "hdgnn_normalize_propagate_backward": dict(W=None, out=None, dH=None, dW=None, dbias=None),
            "hdgnn_map_conv_backward": dict(dx=None, dtheta=None, work=None)}


def _validates(fn):
    """Every bad case of `fn` is refused with a message naming the entry point and the argument; without a GPU, valid arguments
    (with and without the optional pointers) reach the device and fail loudly there."""
    names, valid, bad = TABLE[fn]
    for change in bad:
        assert getattr(lib, fn)(*_args(names, valid, change), None) == E_INVALID, change
        msg = lib.hdgnn_last_error(None).decode()
        assert msg.startswith(fn + ": ") and next(iter(change)) in msg[len(fn) + 2:], (change, msg)
    if not torch.cuda.is_available():                # fake pointers must never reach a real device
        for change in ({}, OPTIONAL[fn]):
            assert getattr(lib, fn)(*_args(names, valid, change), None) == E_CUDA, change
            assert lib.hdgnn_last_error(None).decode().startswith(fn + ": ")


def test_hunk_groups_validates_arguments_without_a_gpu():
    _validates("hdgnn_hunk_groups")


def test_partition_counts_validates_arguments_without_a_gpu():
    _validates("hdgnn_partition_counts")


def test_hunk_clusters_validates_arguments_without_a_gpu():
    _validates("hdgnn_hunk_clusters")
    work_of = lib.hdgnn_hunk_clusters_work
    # the two tables of a commit live in shared memory up to n = 169, above that in one slice of the workspace per CTA
    assert work_of(100, 74) == 0 and work_of(100, 169) == 0
    assert work_of(100, 170) == 100 * 2 * 170 * 171 * 4 and work_of(4096, 512) == 296 * 2 * 512 * 513 * 4
    assert work_of(0, 300) == 0 and work_of(1, 513) == 0 and work_of(1, 1) == 0


def test_compact_from_raw_validates_arguments_without_a_gpu():
    _validates("hdgnn_compact_from_raw")


def test_eval_counts_validates_arguments_without_a_gpu():
    _validates("hdgnn_eval_counts")


def test_pack_label_bits_validates_arguments_without_a_gpu():
    _validates("hdgnn_pack_label_bits")


def test_normalize_propagate_validates_arguments_without_a_gpu():
    _validates("hdgnn_normalize_propagate")


def test_map_conv_validates_arguments_without_a_gpu():
    _validates("hdgnn_map_conv")


def test_normalize_propagate_backward_validates_arguments_without_a_gpu():
    _validates("hdgnn_normalize_propagate_backward")


def test_map_conv_backward_validates_arguments_without_a_gpu():
    _validates("hdgnn_map_conv_backward")


def _c_calls(N, adj_ptr, pitch, flags):
    """The four legacy entry points with fake device pointers -> {name: (return code, message)}: each must refuse the adjacency
    before any CUDA call."""
    f = C.c_void_p(1 << 20)
    calls = {
        "normalize_propagate": lambda: lib.hdgnn_normalize_propagate(2, N, adj_ptr, pitch, f, 20, None, None, 20, 1e-3, flags, f, None,
                                                                     None),
        "map_conv": lambda: lib.hdgnn_map_conv(2, N, adj_ptr, pitch, f, f, 1.5, 1e-3, flags, f, None, None),
        "normalize_propagate_backward": lambda: lib.hdgnn_normalize_propagate_backward(2, N, adj_ptr, pitch, f, 20, None, 20, 1e-3,
                                                                                      flags, None, f, f, None, None, f, None),
        "map_conv_backward": lambda: lib.hdgnn_map_conv_backward(2, N, adj_ptr, pitch, f, f, 1.5, 1e-3, flags, 1.0, f, None, None,
                                                                 None),
    }
    return {name: (call(), lib.hdgnn_last_error(None).decode()) for name, call in calls.items()}


@pytest.mark.parametrize("N", [9, 200, 512])
def test_bitmap_pitch_and_alignment_are_checked_before_launch(N):
    from hdgnn_b200.engine import P_LABEL_BITS, bit_words, label_pitch
    aligned, pitch = C.c_void_p(1 << 24), 4 * bit_words(N)
    wrong = {label_pitch(N), pitch + 16, pitch - 16, 4 * ((N + 31) // 32)} - {pitch, 0}     # byte pitch, unpadded rows, ...
    bad = [(aligned, p) for p in sorted(wrong)] + [(C.c_void_p((1 << 24) + 4), pitch)]      # ... and a misaligned base
    for adj, p in bad:
        for name, (rc, msg) in _c_calls(N, adj, p, P_LABEL_BITS).items():
            assert rc == E_INVALID and msg.startswith(f"hdgnn_{name}: adj"), (name, p, adj.value, msg)
    for name, (rc, msg) in _c_calls(_lib.MAX_N + 1, aligned, 4 * 16, P_LABEL_BITS).items():
        assert rc == E_INVALID and msg.startswith(f"hdgnn_{name}: N"), (name, msg)


# ---- the Python wrappers -------------------------------------------------------------------------------------------------
def _wrapper_calls():
    """(wrapper, call with one wrong shape, call with right shapes) on CPU tensors."""
    from hdgnn_b200 import engine as E
    B, N, n = 2, 40, 30
    adj, bits = torch.zeros(B, N, 48, dtype=torch.uint8), torch.zeros(B, N, E.bit_words(N), dtype=torch.int32)
    H, x, th = torch.zeros(B, N, 20), torch.zeros(B, N), torch.zeros(2)
    probs, Y = torch.zeros(B, 2, n * (n - 1)), torch.zeros(B, n, 32, dtype=torch.uint8)
    lab, nh = torch.zeros(B, n, dtype=torch.int32), torch.zeros(B, dtype=torch.int32)
    return [
        ("normalize_propagate H", lambda: E.normalize_propagate(adj, H[:, :-1]), lambda: E.normalize_propagate(bits, H)),
        ("normalize_propagate W", lambda: E.normalize_propagate(adj, H, torch.zeros(19, 8)), lambda: E.normalize_propagate(adj, H, torch.zeros(20, 8))),
        ("normalize_propagate bias", lambda: E.normalize_propagate(adj, H, torch.zeros(20, 8), torch.zeros(20)),
         lambda: E.normalize_propagate(adj, H, torch.zeros(20, 8), torch.zeros(8))),
        ("map_conv x", lambda: E.map_conv(bits, x[:1], th), lambda: E.map_conv(bits, x, th)),
        ("map_conv theta", lambda: E.map_conv(adj, x, torch.zeros(3)), lambda: E.map_conv(adj, x, th[None])),
        ("normalize_propagate_backward dOut", lambda: E.normalize_propagate_backward(adj, H, H[:1]),
         lambda: E.normalize_propagate_backward(adj, H, H)),
        ("normalize_propagate_backward out", lambda: E.normalize_propagate_backward(adj, H, H, out=H[:, :, :4], flags=E.P_RELU),
         lambda: E.normalize_propagate_backward(adj, H, H, out=H, flags=E.P_RELU)),
        ("normalize_propagate_backward H", lambda: E.normalize_propagate_backward(bits, H[:, :3], H),
         lambda: E.normalize_propagate_backward(bits, H, H)),
        ("normalize_propagate_backward W", lambda: E.normalize_propagate_backward(adj, H, H[..., :8], W=torch.zeros(20, 20)),
         lambda: E.normalize_propagate_backward(adj, H, H[..., :8], W=torch.zeros(20, 8))),
        ("map_conv_backward x", lambda: E.map_conv_backward(adj, x[:, :-1], th), lambda: E.map_conv_backward(adj, x, th)),
        ("map_conv_backward theta", lambda: E.map_conv_backward(adj, x, th[:1]), lambda: E.map_conv_backward(adj, x, th)),
        ("compact_from_raw_device", lambda: E.compact_from_raw_device(torch.zeros(B, n, n + 1, dtype=torch.float64)),
         lambda: E.compact_from_raw_device(torch.zeros(B, n, n, dtype=torch.float64))),
        ("pack_label_bits_device", lambda: E.pack_label_bits_device(Y[0]), lambda: E.pack_label_bits_device(Y)),
        ("eval_counts", lambda: E.eval_counts(probs[:, :, 1:], Y), lambda: E.eval_counts(probs, Y)),
        ("hunk_groups", lambda: E.hunk_groups(bits[:, :, :-1]), lambda: E.hunk_groups(bits)),
        ("partition_counts truth", lambda: E.partition_counts(lab, lab[:1]), lambda: E.partition_counts(lab, lab)),
        ("partition_counts nh", lambda: E.partition_counts(lab, lab, nh[:1]), lambda: E.partition_counts(lab, lab, nh)),
        ("hunk_clusters probs", lambda: E.hunk_clusters(probs[:, :, 1:]), lambda: E.hunk_clusters(probs)),
        ("hunk_clusters nh", lambda: E.hunk_clusters(probs, nh[:1]), lambda: E.hunk_clusters(probs, nh)),
    ]


@pytest.mark.parametrize("case", range(len(_wrapper_calls())))
def test_wrappers_reject_wrong_shapes_before_the_cuda_check(case):
    what, wrong, right = _wrapper_calls()[case]
    with pytest.raises(ValueError):
        wrong()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        right()


# ---- on the GPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusal_carries_its_own_message_not_an_earlier_create_error():
    from hdgnn_b200.engine import Engine, bit_words, map_conv
    with pytest.raises(_lib.HdgnnError):
        Engine(600, 10)                                                 # leaves a create error on this thread
    create_msg = lib.hdgnn_last_error(None).decode()
    assert create_msg
    N = 200
    flat = torch.zeros(N * bit_words(N) + 1, dtype=torch.int32, device="cuda")
    with pytest.raises(_lib.HdgnnError) as e:
        map_conv(flat[1:].view(1, N, bit_words(N)), torch.zeros(1, N, device="cuda"), torch.zeros(2, device="cuda"))
    assert e.value.code == E_INVALID
    assert "hdgnn_map_conv: adj" in str(e.value) and create_msg not in str(e.value)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two devices")
def test_tensors_on_two_devices_are_refused():
    from hdgnn_b200.engine import eval_counts, hunk_clusters, map_conv, partition_counts
    n = 30
    lab0, lab1 = torch.zeros(2, n, dtype=torch.int32, device="cuda:0"), torch.zeros(2, n, dtype=torch.int32, device="cuda:1")
    probs1 = torch.zeros(2, 2, n * (n - 1), device="cuda:1")
    with pytest.raises(ValueError, match="one device"):
        partition_counts(lab0, lab1)
    with pytest.raises(ValueError, match="one device"):
        hunk_clusters(probs1, torch.full((2,), n, dtype=torch.int32, device="cuda:0"))
    with pytest.raises(ValueError, match="one device"):
        eval_counts(probs1, torch.zeros(2, n, 32, dtype=torch.uint8, device="cuda:0"))
    with pytest.raises(ValueError, match="one device"):
        map_conv(torch.zeros(2, n, 32, dtype=torch.uint8, device="cuda:1"), torch.zeros(2, n, device="cuda:0"),
                 torch.zeros(2, device="cuda:1"))
