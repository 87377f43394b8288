"""Host-side engine: owns one libhdgnn handle and feeds it torch CUDA tensors by pointer.

PyTorch is plumbing here (device memory, streams, torch.distributed); all arithmetic of the hot
path -- model_2.py:86-118 forward, its backward, and the Adam step of model_2.py:336-338 -- runs
in the sm_100a kernels behind the C ABI of include/hdgnn.h.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from ._lib import lib, check

PARAM_NAMES = {
    1: ["hnk_w1", "hnk_b1", "hnk_w2", "hnk_b2", "scr_w1", "scr_b1", "scr_w2", "scr_b2", "theta1", "theta2"],
}
_ENT = ["ent_w1", "ent_b1", "ent_w5", "ent_b5", "nod_w1", "nod_b1", "nod_w2", "nod_b2"]
_EDGE = ["edg_w11", "edg_w12", "edg_b1", "edg_w2", "edg_b2", "eup_w1", "eup_b1", "eup_w2", "eup_b2"]
PARAM_NAMES[2] = _ENT + PARAM_NAMES[1]
PARAM_NAMES[3] = _EDGE + PARAM_NAMES[1]
PARAM_NAMES[4] = _ENT + _EDGE + PARAM_NAMES[1]


def param_count(variant: int) -> int:
    n = lib.hdgnn_param_count(variant)
    if n < 0:
        raise ValueError(f"variant must be 1..4, got {variant}")
    return n


def param_offsets(variant: int) -> Dict[str, int]:
    return {n: lib.hdgnn_param_offset(variant, n.encode()) for n in PARAM_NAMES[variant]}


def label_pitch(n: int) -> int:
    return lib.hdgnn_label_pitch(n)


F_DEBUG, F_LEGACY, F_LABEL_BITS, F_DENSE_SWEEP = 2, 4, 8, 16


def bit_words(n: int) -> int:
    return lib.hdgnn_bit_words(n)


def pack_label_bits(lab: np.ndarray) -> np.ndarray:
    """(B,n,n) {0,1} label grid -> (B,n,bit_words(n)) uint32 bitmap, the wire format of HDGNN_F_LABEL_BITS
    (include/hdgnn.h): word w of a row holds column 32 w + k at bit k; diagonal and padding bits zero."""
    lab = np.asarray(lab)
    B, n, _ = lab.shape
    wp = bit_words(n)
    wide = np.zeros((B, n, wp * 32), dtype=np.uint8)
    wide[:, :, :n] = lab != 0
    wide[:, np.arange(n), np.arange(n)] = 0
    return np.ascontiguousarray(np.packbits(wide, axis=-1, bitorder="little")).view("<u4").reshape(B, n, wp)


@dataclass
class DeviceBatch:
    """Compact commit batch resident in HBM (layouts of include/hdgnn.h)."""
    adj: torch.Tensor    # (B, Ne, pitch_e) uint8
    x: torch.Tensor      # (B, Ne) float32
    hmap: torch.Tensor   # (B, Ne) int32
    L: torch.Tensor      # (B,) int32
    Y: torch.Tensor      # (B, Nc, pitch_c) uint8
    Ne: int
    Nc: int

    @property
    def B(self):
        return self.adj.shape[0]

    @staticmethod
    def from_numpy(adj, x, hmap, L, Y, device, bits: bool = False) -> "DeviceBatch":
        """bits=True: label grids as bitmaps (engines created with F_LABEL_BITS), packed on the device."""
        B, Ne, _ = adj.shape
        Nc = Y.shape[1]
        pe, pc = label_pitch(Ne), label_pitch(Nc)
        a = torch.zeros(B, Ne, pe, dtype=torch.uint8, device=device)
        a[:, :, :Ne] = torch.as_tensor(np.ascontiguousarray(adj, dtype=np.uint8)).to(device)
        y = torch.zeros(B, Nc, pc, dtype=torch.uint8, device=device)
        y[:, :, :Nc] = torch.as_tensor(np.ascontiguousarray(Y, dtype=np.uint8)).to(device)
        if bits:
            a, y = pack_label_bits_device(a), pack_label_bits_device(y)
        return DeviceBatch(
            a, torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)).to(device),
            torch.as_tensor(np.ascontiguousarray(hmap, dtype=np.int32)).to(device),
            torch.as_tensor(np.ascontiguousarray(L, dtype=np.int32)).to(device), y, Ne, Nc)


def pack_label_bits_device(grid: torch.Tensor) -> torch.Tensor:
    """(N,n,pitch) u8 CUDA byte grid (pitch = label_pitch(n)) -> (N,n,bit_words(n)) int32 bitmap (hdgnn_pack_label_bits)."""
    if grid.dim() != 3:
        raise ValueError(f"pack_label_bits_device needs a (N, n, pitch) byte grid, got {tuple(grid.shape)}")
    N, n, pitch = grid.shape
    bits = torch.empty(N, n, bit_words(n), dtype=torch.int32, device=grid.device)
    _launch("pack_label_bits_device", lib.hdgnn_pack_label_bits, N, n, (grid.contiguous(), U8), pitch, bits)
    return bits


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


F32, I32, U8, BITMAP = (torch.float32,), (torch.int32,), (torch.uint8,), (torch.int32, torch.uint32)


def _launch(name: str, fn, *args):
    """Call the stateless libhdgnn entry point `fn` on `args` and the stream.  Tensors are passed by pointer; an input is given
    as (tensor or None, allowed dtypes).  Every tensor must be a CUDA tensor (RuntimeError), all of them on one device and of
    their dtypes (ValueError).  The call runs with that device current, on its current stream; a refusal raises HdgnnError
    with the library's message."""
    want = [a for a in args if isinstance(a, tuple)]
    args = [a[0] if isinstance(a, tuple) else a for a in args]
    tensors = [t for t in args if isinstance(t, torch.Tensor)]
    if not all(t.is_cuda for t in tensors):
        raise RuntimeError(f"{name} needs CUDA tensors; there is no CPU fallback")
    devices = {t.device for t in tensors}
    if len(devices) > 1:
        raise ValueError(f"{name} needs all tensors on one device, got {sorted(map(str, devices))}")
    for t, dtypes in want:
        if t is not None and t.dtype not in dtypes:
            raise ValueError(f"{name} needs {' or '.join(map(str, dtypes))}, got {t.dtype}")
    dev = tensors[0].device
    with torch.cuda.device(dev):
        check(fn(*[_p(a) if isinstance(a, torch.Tensor) else a for a in args], C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))


def _shape(name: str, arg: str, t: Optional[torch.Tensor], *shape):
    """ValueError unless t (None passes) has `shape`; an extent None matches any."""
    if t is not None and (t.dim() != len(shape) or any(s is not None and s != e for s, e in zip(shape, t.shape))):
        want = ", ".join("*" if s is None else str(s) for s in shape)
        raise ValueError(f"{name} needs {arg} of shape ({want}), got {tuple(t.shape)}")


def _f32(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    return None if t is None else t.contiguous().float()


class Engine:
    def __init__(self, Ne: int, Nc: int, variant: int = 2, max_batch: int = 100, device: int = 0,
                 rows_per_cta_e: int = 0, rows_per_cta_c: int = 0, flags: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("hdgnn_b200.Engine needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.Ne, self.Nc, self.variant, self.max_batch, self.device = Ne, Nc, variant, max_batch, device
        self.Ncr = Nc * (Nc - 1)
        self.n_params = param_count(variant)
        cfg = _lib.Config(Ne, Nc, variant, max_batch, device, rows_per_cta_e, rows_per_cta_c, flags)
        h = C.c_void_p()
        check(lib.hdgnn_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.tdev = torch.device("cuda", device)
        self.host_bits = bool(flags & F_LABEL_BITS)      # label grids travel as bitmaps (host and device entry points)
        self._pred_rows = None                           # rows of the set_predictions buffer, None = predictions off
        # row pitch in bytes of the label arrays the device entry points take
        self.pe, self.pc = (4 * bit_words(Ne), 4 * bit_words(Nc)) if self.host_bits else (label_pitch(Ne), label_pitch(Nc))

    def close(self):
        if getattr(self, "_h", None):
            lib.hdgnn_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    def _check_rows(self, B: int):
        assert self._pred_rows is None or B <= self._pred_rows, "the set_predictions buffer has fewer rows than the batch"

    def _check_batch(self, b: DeviceBatch, params: torch.Tensor):
        assert b.Ne == self.Ne and b.Nc == self.Nc, "batch shape does not match the engine"
        self._check_rows(b.B)
        assert params.dtype == torch.float32 and params.is_cuda and params.numel() == self.n_params

    # -- device-resident entry points ---------------------------------------------------------
    def forward(self, b: DeviceBatch, params: torch.Tensor, want_logits=True, want_probs=True):
        """Inference graph of model_2.py:486-502 -> (probs (B,2,Ncr) or None, logits or None, CE scalar tensor).
        want_probs=False: the probabilities are not written (a caller of set_predictions that wants only the bitmap)."""
        self._check_batch(b, params)
        B = b.B
        probs = torch.empty(B, 2, self.Ncr, dtype=torch.float32, device=self.tdev) if want_probs else None
        logits = torch.empty(B, 2, self.Ncr, dtype=torch.float32, device=self.tdev) if want_logits else None
        loss = torch.empty(1, dtype=torch.float32, device=self.tdev)
        check(lib.hdgnn_forward(self._h, B, _p(b.adj), self.pe, _p(b.x), _p(b.hmap), _p(b.L), _p(b.Y), self.pc,
                                _p(params), _p(logits), _p(probs), _p(loss), self._stream()), self._h)
        return probs, logits, loss

    def forward_backward(self, b: DeviceBatch, params: torch.Tensor, B_global: Optional[int] = None,
                         grads: Optional[torch.Tensor] = None, probs: Optional[torch.Tensor] = None,
                         logits: Optional[torch.Tensor] = None, loss: Optional[torch.Tensor] = None,
                         want_probs=True, want_logits=False):
        """-> (probs, logits, loss, grads); grads = d(10*CE)/dparams with CE the mean over B_global*Ncr pairs."""
        self._check_batch(b, params)
        B = b.B
        if probs is None and want_probs:
            probs = torch.empty(B, 2, self.Ncr, dtype=torch.float32, device=self.tdev)
        if logits is None and want_logits:
            logits = torch.empty(B, 2, self.Ncr, dtype=torch.float32, device=self.tdev)
        if loss is None:
            loss = torch.empty(1, dtype=torch.float32, device=self.tdev)
        if grads is None:
            grads = torch.empty(self.n_params, dtype=torch.float32, device=self.tdev)
        check(lib.hdgnn_forward_backward(self._h, B, B if B_global is None else B_global, _p(b.adj), self.pe, _p(b.x),
                                         _p(b.hmap), _p(b.L), _p(b.Y), self.pc, _p(params), _p(logits), _p(probs),
                                         _p(loss), _p(grads), self._stream()), self._h)
        return probs, logits, loss, grads

    def adam_step(self, params, grads, m, v, step_counter, lr=3e-4, beta1=0.9, beta2=0.999, eps=1e-8,
                  reg_losses: Optional[torch.Tensor] = None):
        """Regularisers + tf.train.AdamOptimizer update (model_2.py:121-130, 326-338), in place."""
        check(lib.hdgnn_adam_step(self._h, _p(params), _p(grads), _p(m), _p(v), _p(step_counter), lr, beta1, beta2,
                                  eps, _p(reg_losses), self._stream()), self._h)

    def train_step(self, b: DeviceBatch, params, m, v, step_counter, loss3, probs=None, logits=None,
                   lr=3e-4, beta1=0.9, beta2=0.999, eps=1e-8):
        """One fused training step on one GPU (forward, backward, regularisers, TF1 Adam): the body of
        sess.run([..., trainer]) of model_2.py:369-383.  loss3 (3,) receives {CE, loss_map, loss_para}."""
        self._check_batch(b, params)
        check(lib.hdgnn_train_step(self._h, b.B, _p(b.adj), self.pe, _p(b.x), _p(b.hmap), _p(b.L), _p(b.Y), self.pc,
                                   _p(params), _p(m), _p(v), _p(step_counter), lr, beta1, beta2, eps,
                                   _p(logits), _p(probs), _p(loss3), self._stream()), self._h)

    # -- host-buffer entry points (H2D + compute + D2H on one stream) -----------------------------
    def train_step_host(self, adj, x, hmap, L, Y, params, m, v, step_counter, loss3, probs=None,
                        lr=3e-4, beta1=0.9, beta2=0.999, eps=1e-8):
        """adj (B,Ne,Ne) u8, x (B,Ne) f32, hmap (B,Ne) i32, L (B,) i32, Y (B,Nc,Nc) u8: pinned host
        tensors (adj / Y as pack_label_bits bitmaps when the engine was created with F_LABEL_BITS);
        loss3 (3,) pinned float32 receives {CE, loss_map, loss_para}.  Asynchronous."""
        B = adj.shape[0]
        self._check_rows(B)
        check(lib.hdgnn_train_step_host(self._h, B, _p(adj), _p(x), _p(hmap), _p(L), _p(Y), _p(params), _p(m), _p(v),
                                        _p(step_counter), lr, beta1, beta2, eps, _p(probs), _p(loss3),
                                        self._stream()), self._h)

    def forward_backward_host(self, adj, x, hmap, L, Y, params, grads, B_global, loss=None, probs=None):
        """Commit-sharded training from pinned host tensors: H2D + forward + backward; grads / loss / probs on device."""
        B = adj.shape[0]
        self._check_rows(B)
        check(lib.hdgnn_forward_backward_host(self._h, B, B_global, _p(adj), _p(x), _p(hmap), _p(L), _p(Y), _p(params),
                                              _p(probs), _p(loss), _p(grads), self._stream()), self._h)

    # -- commit sharding with the all-reduce fused into the last kernel (peer memory over NVLink) ----------------
    def peer_attach(self, collective: str = "peer") -> bool:
        """Exchange the CUDA IPC handles of the ranks' mailboxes through torch.distributed and map them
        (hdgnn_peer_export / hdgnn_peer_attach).  Collective call.  Returns True when every rank is attached; with
        collective="auto" a failure on any rank (multi-kernel path, no P2P) returns False on all ranks instead of raising."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()
        buf = (C.c_ubyte * 64)()
        rc = lib.hdgnn_peer_export(self._h, world, buf) if 2 <= world <= 8 else _lib.E_UNSUPPORTED
        flag = torch.tensor([1 if rc == _lib.OK else 0], device=self.tdev, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if not int(flag.item()):
            if collective == "auto":
                return False
            check(rc if rc != _lib.OK else _lib.E_UNSUPPORTED, self._h)
        handles = [None] * world
        dist.all_gather_object(handles, bytes(buf))
        rc = lib.hdgnn_peer_attach(self._h, rank, world, b"".join(handles))
        flag = torch.tensor([1 if rc == _lib.OK else 0], device=self.tdev, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)          # also the barrier the first exchange needs
        if not int(flag.item()):
            if collective == "auto":
                return False
            check(rc if rc != _lib.OK else _lib.E_CUDA, self._h)
        self.peer_world = world
        return True

    def set_hits_accumulator(self, acc: Optional[torch.Tensor]) -> bool:
        """acc: one-element int64 CUDA tensor that every later step adds its arg-max hits to (None: off).  Returns False when
        this engine runs the multi-kernel path, which has no in-kernel counter (use eval_counts)."""
        rc = lib.hdgnn_set_hits_accumulator(self._h, _p(acc))
        if rc == _lib.E_UNSUPPORTED:
            return False
        check(rc, self._h)
        self._hits_ref = acc            # keep the tensor alive while the handle points at it
        return True

    def set_eval_counters(self, counts: Optional[torch.Tensor]) -> bool:
        """counts: (B, 8) int64 CUDA tensor (layout of eval_counts) that the relation head of every later forward / training call
        adds the commits' evaluation counters to (None: off).  Returns False on the multi-kernel path (use eval_counts)."""
        if counts is not None:
            assert counts.dtype == torch.int64 and counts.is_cuda and counts.is_contiguous() and counts.shape[-1] == 8
        rc = lib.hdgnn_set_eval_counters(self._h, _p(counts))
        if rc == _lib.E_UNSUPPORTED:
            return False
        check(rc, self._h)
        self._evc_ref = counts          # keep the tensor alive while the handle points at it
        return True

    def set_predictions(self, bits: Optional[torch.Tensor]):
        """bits: (B, Nc, bit_words(Nc)) int32 CUDA tensor that the relation head of every later forward / training call WRITES the
        commits' predicted relations to, as a label bitmap (bit (s,t) = [p1 > p0], the arg-max; hdgnn_set_predictions); row b is
        commit b of a call, so B must cover the batch size of every call made while it is set.  None: off."""
        if bits is not None:
            assert bits.dtype == torch.int32 and bits.is_cuda and bits.is_contiguous()
            assert bits.dim() == 3 and bits.shape[1:] == (self.Nc, bit_words(self.Nc))
        self._pred_rows = None if bits is None else bits.shape[0]
        check(lib.hdgnn_set_predictions(self._h, _p(bits)), self._h)
        self._pred_ref = bits           # keep the tensor alive while the handle points at it

    def peer_status(self):
        """Raises HdgnnError(E_PEER) if a gradient exchange timed out since peer_attach (synchronises with the device)."""
        check(lib.hdgnn_peer_status(self._h), self._h)

    def train_step_peer(self, b: DeviceBatch, params, m, v, step_counter, loss3, probs=None, logits=None,
                        lr=3e-4, beta1=0.9, beta2=0.999, eps=1e-8):
        """This rank's shard of one training step; gradients are exchanged inside the last kernel (no NCCL call)."""
        self._check_batch(b, params)
        check(lib.hdgnn_train_step_peer(self._h, b.B, b.B * self.peer_world, _p(b.adj), self.pe, _p(b.x), _p(b.hmap), _p(b.L),
                                        _p(b.Y), self.pc, _p(params), _p(m), _p(v), _p(step_counter), lr, beta1, beta2, eps,
                                        _p(logits), _p(probs), _p(loss3), self._stream()), self._h)

    def train_step_peer_host(self, adj, x, hmap, L, Y, params, m, v, step_counter, loss3, probs=None,
                             lr=3e-4, beta1=0.9, beta2=0.999, eps=1e-8):
        B = adj.shape[0]
        self._check_rows(B)
        check(lib.hdgnn_train_step_peer_host(self._h, B, B * self.peer_world, _p(adj), _p(x), _p(hmap), _p(L), _p(Y), _p(params),
                                             _p(m), _p(v), _p(step_counter), lr, beta1, beta2, eps, _p(probs), _p(loss3),
                                             self._stream()), self._h)

    def infer_host(self, adj, x, hmap, L, Y, params, probs=None, loss=None):
        """Inference from pinned host tensors (layouts of train_step_host).  probs: host or device tensor (B, 2, Ncr), or None
        when only the predictions (set_predictions), the counters (set_eval_counters) or the loss are wanted."""
        B = adj.shape[0]
        self._check_rows(B)
        check(lib.hdgnn_infer_host(self._h, B, _p(adj), _p(x), _p(hmap), _p(L), _p(Y), _p(params), _p(probs),
                                   _p(loss), self._stream()), self._h)

    # -- introspection ------------------------------------------------------------------------------
    def workspace(self, name: str, shape, dtype=torch.float32) -> torch.Tensor:
        """Copy of a named scratch buffer (tests only)."""
        n = int(np.prod(shape))
        out = torch.empty(n, dtype=dtype, device=self.tdev)
        check(lib.hdgnn_workspace_copy(self._h, name.encode(), _p(out), n * out.element_size(), self._stream()),
              self._h)
        torch.cuda.current_stream(self.tdev).synchronize()
        return out.reshape(shape)

    def profile(self, enable: bool):
        check(lib.hdgnn_profile(self._h, 1 if enable else 0), self._h)

    def profile_records(self):
        """[(kernel label, milliseconds)] of every launch since profile(True)."""
        out = []
        buf = C.create_string_buffer(64)
        ms = C.c_float()
        for i in range(lib.hdgnn_profile_count(self._h)):
            check(lib.hdgnn_profile_get(self._h, i, buf, 64, C.byref(ms)), self._h)
            out.append((buf.value.decode(), ms.value))
        return out

    def last_launch_count(self) -> int:
        return lib.hdgnn_last_launch_count(self._h)


# -- legacy operator of model.py (normalize_adj + propagation, Chebyshev map_conv) -------------------------------
P_SELF_LOOP, P_RELU, P_NO_TRANSPOSE, P_NO_TENSOR, P_TENSOR_V1, P_LABEL_BITS = 1, 2, 4, 8, 16, 32


def _pitched(adj: torch.Tensor) -> torch.Tensor:
    """(B,N,N) uint8 cuda -> (B,N,pitch) with the row pitch the kernels need."""
    B, N, M = adj.shape
    pitch = label_pitch(N)
    if M == pitch:
        return adj.contiguous()
    out = torch.zeros(B, N, pitch, dtype=torch.uint8, device=adj.device)
    out[:, :, :N] = adj[:, :, :N]
    return out


def _adjacency(adj: torch.Tensor, flags: int):
    """The legacy operator's adjacency argument -> (tensor, row pitch in bytes, flags).  An int32 / uint32 tensor is a label
    bitmap (B,N,bit_words(N)) as pack_label_bits_device returns it and sets P_LABEL_BITS; a uint8 tensor is a byte grid."""
    if adj.dtype in (torch.int32, torch.uint32):
        B, N, wp = adj.shape
        if wp != bit_words(N):
            raise ValueError(f"a label bitmap of N = {N} has bit_words(N) = {bit_words(N)} words per row, got {wp}")
        return adj.contiguous(), 4 * wp, flags | P_LABEL_BITS
    if flags & P_LABEL_BITS:
        raise ValueError("P_LABEL_BITS needs an int32 / uint32 label bitmap, got a byte grid")
    a = _pitched(adj)
    return a, a.shape[2], flags


def normalize_propagate(adj: torch.Tensor, H: torch.Tensor, W: Optional[torch.Tensor] = None,
                        bias: Optional[torch.Tensor] = None, eps: float = 1e-3, flags: int = 0):
    """act(A_hat (H W) + b) with the reference's normalize_adj (model.py:360-367).  adj (B,N,N|pitch) uint8 cuda, or a
    (B,N,bit_words(N)) int32 / uint32 label bitmap (the same operator, P_LABEL_BITS is set here), H (B,N,d_in) float32
    cuda.  Returns (out (B,N,d_out), dinv (B,N))."""
    name = "normalize_propagate"
    a, pitch, flags = _adjacency(adj, flags)
    B, N = a.shape[:2]
    _shape(name, "H", H, B, N, None)
    d_in = H.shape[2]
    _shape(name, "W", W, d_in, None)
    d_out = d_in if W is None else W.shape[1]
    _shape(name, "bias", bias, d_out)
    out = torch.empty(B, N, d_out, dtype=torch.float32, device=a.device)
    dinv = torch.empty(B, N, dtype=torch.float32, device=a.device)
    _launch(name, lib.hdgnn_normalize_propagate, B, N, a, pitch, _f32(H), d_in, _f32(W), _f32(bias), d_out, eps, flags, out, dinv)
    return out, dinv


def map_conv(adj: torch.Tensor, x: torch.Tensor, theta: torch.Tensor, lam_max: float = 1.5, eps: float = 1e-3,
             flags: int = 0):
    """map_conv of model.py:394-403 (k = 2, Ds = 1); adj as for normalize_propagate.  Returns (loss scalar tensor,
    per-commit (B,))."""
    a, pitch, flags = _adjacency(adj, flags)
    B, N = a.shape[:2]
    _shape("map_conv", "x", x, B, N)
    _shape("map_conv", "theta", theta.reshape(-1), 2)
    per = torch.empty(B, dtype=torch.float32, device=a.device)
    loss = torch.empty(1, dtype=torch.float32, device=a.device)
    _launch("map_conv", lib.hdgnn_map_conv, B, N, a, pitch, _f32(x), _f32(theta.reshape(-1)), lam_max, eps, flags, per, loss)
    return loss, per


def normalize_propagate_backward(adj: torch.Tensor, H: torch.Tensor, dOut: torch.Tensor, W: Optional[torch.Tensor] = None,
                                 out: Optional[torch.Tensor] = None, eps: float = 1e-3, flags: int = 0):
    """Backward of normalize_propagate w.r.t. H, W and the bias (the adjacency carries no gradient: model.py:337 takes its
    argmax); adj as for normalize_propagate.  `out` = the forward's output, needed with P_RELU.  Returns (dH (B,N,d_in),
    dW (d_in,d_out) or None, dbias (d_out))."""
    name = "normalize_propagate_backward"
    a, pitch, flags = _adjacency(adj, flags)
    B, N = a.shape[:2]
    _shape(name, "H", H, B, N, None)
    _shape(name, "dOut", dOut, B, N, None)
    d_in, d_out = H.shape[2], dOut.shape[2]
    _shape(name, "W", W, d_in, d_out)
    _shape(name, "out", out, B, N, d_out)
    dH = torch.empty(B, N, d_in, dtype=torch.float32, device=a.device)
    dW = torch.empty(d_in, d_out, dtype=torch.float32, device=a.device) if W is not None else None
    db = torch.empty(d_out, dtype=torch.float32, device=a.device)
    work = torch.empty(lib.hdgnn_propagate_backward_work(B, N, d_in, d_out), dtype=torch.float32, device=a.device)
    _launch(name, lib.hdgnn_normalize_propagate_backward, B, N, a, pitch, _f32(H), d_in, _f32(W), d_out, eps, flags, _f32(out),
            _f32(dOut), dH, dW, db, work)
    return dH, dW, db


def map_conv_backward(adj: torch.Tensor, x: torch.Tensor, theta: torch.Tensor, lam_max: float = 1.5, eps: float = 1e-3,
                      flags: int = 0, gscale: float = 1.0):
    """Gradient of map_conv's loss w.r.t. x (B,N) and theta (2) (model.py:394-403; no gradient to the adjacency); adj as
    for normalize_propagate."""
    a, pitch, flags = _adjacency(adj, flags)
    B, N = a.shape[:2]
    _shape("map_conv_backward", "x", x, B, N)
    _shape("map_conv_backward", "theta", theta.reshape(-1), 2)
    dx = torch.empty(B, N, dtype=torch.float32, device=a.device)
    dth = torch.empty(2, dtype=torch.float32, device=a.device)
    work = torch.empty(2 * B, dtype=torch.float32, device=a.device)
    _launch("map_conv_backward", lib.hdgnn_map_conv_backward, B, N, a, pitch, _f32(x), _f32(theta.reshape(-1)), lam_max, eps, flags,
            gscale, dx, dth, work)
    return dx, dth


# -- data formats either side of the hot path: device loader and device evaluation (SURVEY 8(f) rows 1, 2) --------
def compact_from_raw_device(raw: torch.Tensor, want_diag: bool = True):
    """utils2.py:29-47 + the int() label indexing of :82,:105 on the device.  raw: (N,n,n) float64 / float32 CUDA tensor
    as stored in CAdjs / CHunkAdjs.  Returns (grid u8 (N,n,pitch), diag f32 (N,n) or None); raises IndexError where
    the reference would (an off-diagonal entry that does not truncate to -2, -1, 0 or 1)."""
    if raw.dim() != 3 or raw.shape[1] != raw.shape[2]:
        raise ValueError(f"compact_from_raw_device needs raw of shape (N, n, n), got {tuple(raw.shape)}")
    N, n, _ = raw.shape
    if raw.dtype not in (torch.float64, torch.float32):
        raw = raw.to(torch.float64)
    pitch = label_pitch(n)
    grid = torch.empty(N, n, pitch, dtype=torch.uint8, device=raw.device)
    diag = torch.empty(N, n, dtype=torch.float32, device=raw.device) if want_diag else None
    err = torch.zeros(1, dtype=torch.int32, device=raw.device)
    _launch("compact_from_raw_device", lib.hdgnn_compact_from_raw, N, n, raw.contiguous(), 1 if raw.dtype == torch.float64 else 0,
            grid, pitch, diag, err)
    if int(err.item()):
        raise IndexError("off-diagonal entries must truncate to 0 or 1 (utils2.py:82,105)")
    return grid, diag


def eval_counts(probs: torch.Tensor, Y: torch.Tensor, auc: bool = False, auc_first: int = 0):
    """Evaluation counters of EvaluationFuncs.py on the device.  probs (B,2,Ncr) f32 CUDA, Y (B,Nc,Nc|pitch) u8 CUDA.
    Returns (counts (B,8) int64, auc (B,2) int64 or None), see include/hdgnn.h; feed them to
    EvaluationFuncs.metrics_from_counts."""
    _shape("eval_counts", "Y", Y, None, None, None)
    B, Nc, pitch = Y.shape
    _shape("eval_counts", "probs", probs, B, 2, Nc * (Nc - 1))
    counts = torch.empty(B, 8, dtype=torch.int64, device=probs.device)
    a = torch.empty(B, 2, dtype=torch.int64, device=probs.device) if auc else None
    _launch("eval_counts", lib.hdgnn_eval_counts, B, Nc, (probs.contiguous(), F32), (Y.contiguous(), U8), pitch, counts, a, auc_first)
    return counts, a


def hunk_groups(bits: torch.Tensor):
    """Hunk groups of label bitmaps (hdgnn_hunk_groups): bits (B, n, bit_words(n)) int32 CUDA tensor, e.g. what set_predictions
    receives, or the labels.  Hunks s and t share a group when bit (s,t) or bit (t,s) is set.  Returns (groups (B, n) int32: the
    smallest hunk index of each hunk's group, ngroups (B,) int32)."""
    if bits.dim() != 3 or bits.shape[2] != bit_words(bits.shape[1]):
        raise ValueError(f"hunk_groups needs a (B, n, bit_words(n)) label bitmap, got {tuple(bits.shape)}")
    B, n, _ = bits.shape
    groups = torch.empty(B, n, dtype=torch.int32, device=bits.device)
    ngroups = torch.empty(B, dtype=torch.int32, device=bits.device)
    _launch("hunk_groups", lib.hdgnn_hunk_groups, B, n, (bits.contiguous(), BITMAP), groups, ngroups)
    return groups, ngroups


def partition_counts(pred: torch.Tensor, truth: torch.Tensor, nh: Optional[torch.Tensor] = None):
    """Partition-agreement counters of two hunk groupings per commit (hdgnn_partition_counts), e.g. hunk_groups of the predicted
    relations and of the labels: pred, truth (B, n) int32 CUDA tensors, any labels in [0, n) on the real hunks; nh (B,) int32
    CUDA tensor, the number of real hunks of each commit (hunks >= nh[b] are ignored), or None: all n.  Returns counts (B, 8)
    int64 = {real hunks, pairs joined in both, by pred, by truth, groups of pred, of truth, sum of largest overlaps of the pred
    groups, of the truth groups}; a row of -1 marks a commit with nh outside [0, n] or a real hunk labelled outside [0, n).
    Feed them to EvaluationFuncs.partition_metrics_from_counts."""
    _shape("partition_counts", "pred", pred, None, None)
    B, n = pred.shape
    _shape("partition_counts", "truth", truth, B, n)
    _shape("partition_counts", "nh", nh, B)
    counts = torch.empty(B, 8, dtype=torch.int64, device=pred.device)
    _launch("partition_counts", lib.hdgnn_partition_counts, B, n, (pred.contiguous(), I32), (truth.contiguous(), I32),
            (None if nh is None else nh.contiguous(), I32), counts)
    return counts


def hunk_clusters(probs: torch.Tensor, nh: Optional[torch.Tensor] = None, threshold: float = 0.5):
    """Hunk groups by average-linkage clustering of the relation probabilities (hdgnn_hunk_clusters): probs (B, 2, n(n-1))
    float32 CUDA tensor as the relation head writes it (only channel 1 is read); nh (B,) int32 CUDA tensor, the number of real
    hunks of each commit, or None: all n.  Two groups merge while the mean of max(p1(s,t), p1(t,s)) over their hunk pairs is
    > threshold, the closest first.  Returns (groups (B, n) int32: the smallest hunk index of each real hunk's group, s for a
    hunk s >= nh[b]; ngroups (B,) int32), the labelling of hunk_groups; a commit with nh outside [0, n] gets -1 throughout."""
    B, n = _probs_shape("hunk_clusters", probs, nh)
    groups = torch.empty(B, n, dtype=torch.int32, device=probs.device)
    ngroups = torch.empty(B, dtype=torch.int32, device=probs.device)
    nwork = lib.hdgnn_hunk_clusters_work(B, n)
    work = torch.empty(nwork, dtype=torch.uint8, device=probs.device) if nwork else None
    _launch("hunk_clusters", lib.hdgnn_hunk_clusters, B, n, (probs.contiguous(), F32), (None if nh is None else nh.contiguous(), I32),
            float(threshold), groups, ngroups, work)
    return groups, ngroups


def _probs_shape(name: str, probs: torch.Tensor, nh: Optional[torch.Tensor]):
    """(B, n) of relation-head probabilities (B, 2, n(n-1)) with nh (B,) or None; ValueError otherwise."""
    _shape(name, "probs", probs, None, 2, None)
    B, _, ncr = probs.shape
    n = (1 + int(round((1 + 4 * ncr) ** 0.5))) // 2
    if n < 2 or n * (n - 1) != ncr:
        raise ValueError(f"{name} needs n(n-1) pairs per channel, got {ncr}")
    _shape(name, "nh", nh, B)
    return B, n


def hunk_linkage(probs: torch.Tensor, nh: Optional[torch.Tensor] = None):
    """The dendrogram of hunk_clusters (hdgnn_hunk_linkage): the same average-linkage merges on the same inputs, without a
    threshold.  Returns (merges (B, n-1, 2) int32: row i = (a, c), a < c, cluster c joined cluster a; heights (B, n-1) float32:
    the mean of w over the two clusters at that merge; nmerges (B,) int32: the rows recorded, m - 1 unless NaN means were left,
    -1 for a commit with nh outside [0, n]).  Rows past nmerges hold (-1, -1) and NaN.  linkage_cut turns it into groups;
    scipy_linkage into scipy's linkage matrix."""
    B, n = _probs_shape("hunk_linkage", probs, nh)
    merges = torch.empty(B, n - 1, 2, dtype=torch.int32, device=probs.device)
    heights = torch.empty(B, n - 1, dtype=torch.float32, device=probs.device)
    nmerges = torch.empty(B, dtype=torch.int32, device=probs.device)
    nwork = lib.hdgnn_hunk_clusters_work(B, n)
    work = torch.empty(nwork, dtype=torch.uint8, device=probs.device) if nwork else None
    _launch("hunk_linkage", lib.hdgnn_hunk_linkage, B, n, (probs.contiguous(), F32), (None if nh is None else nh.contiguous(), I32),
            merges, heights, nmerges, work)
    return merges, heights, nmerges


def linkage_cut(merges: torch.Tensor, heights: torch.Tensor, nmerges: torch.Tensor, nh: Optional[torch.Tensor] = None,
                thresholds=None, target: Optional[torch.Tensor] = None):
    """Hunk groups from hunk_linkage's record (hdgnn_linkage_cut), at each of `thresholds` (a sequence of 1 to 64 floats: the
    longest prefix of merges whose heights are all > t, which is exactly hunk_clusters(probs, nh, t)) or at `target` ((B,) int32
    CUDA tensor: the merges that leave max(target, 1) groups of the real hunks, or all of them); exactly one of the two.
    Returns (groups (K, B, n) int32, ngroups (K, B) int32) in hunk_clusters' labelling (K = 1 with target); a commit whose
    record is inconsistent gets -1 throughout."""
    if (thresholds is None) == (target is None):
        raise ValueError("linkage_cut needs exactly one of thresholds and target")
    _shape("linkage_cut", "merges", merges, None, None, 2)
    B, n = merges.shape[0], merges.shape[1] + 1
    _shape("linkage_cut", "heights", heights, B, n - 1)
    _shape("linkage_cut", "nmerges", nmerges, B)
    _shape("linkage_cut", "nh", nh, B)
    _shape("linkage_cut", "target", target, B)
    host = None
    if thresholds is not None:
        thresholds = [float(t) for t in thresholds]
        host = (C.c_float * max(len(thresholds), 1))(*thresholds)
    K = 1 if thresholds is None else len(thresholds)
    groups = torch.empty(K, B, n, dtype=torch.int32, device=merges.device)
    ngroups = torch.empty(K, B, dtype=torch.int32, device=merges.device)
    _launch("linkage_cut", lib.hdgnn_linkage_cut, B, n, (merges.contiguous(), I32), (heights.contiguous(), F32),
            (nmerges.contiguous(), I32), (None if nh is None else nh.contiguous(), I32), K, host,
            (None if target is None else target.contiguous(), I32), groups, ngroups)
    return groups, ngroups


def scipy_linkage(merges, heights, nmerges, nh=None) -> list:
    """hunk_linkage's record (tensors or arrays) as scipy's linkage matrices, one per commit: Z (m-1, 4) float64, row i =
    [id of a's cluster, id of c's cluster, 1 - height, size of the new cluster], where a singleton s has id s and the cluster
    formed at row i has id m + i, as scipy.cluster.hierarchy.linkage numbers them; dendrogram and fcluster(Z, 1 - t,
    "distance") then work on the device's result.  ValueError for a commit whose sequence did not join all m real hunks
    (NaN means left over, or nmerges -1)."""
    merges, heights, nmerges = (np.asarray(x.cpu() if torch.is_tensor(x) else x) for x in (merges, heights, nmerges))
    n = merges.shape[1] + 1
    out = []
    for b in range(merges.shape[0]):
        m = n if nh is None else int(np.asarray(nh.cpu() if torch.is_tensor(nh) else nh)[b])
        if int(nmerges[b]) != max(m - 1, 0):
            raise ValueError(f"commit {b}: {int(nmerges[b])} merges of {m} hunks do not form one tree")
        ident = np.arange(max(m, 0))                         # scipy id of the cluster each representative stands for
        size = np.ones(max(m, 0), np.int64)
        Z = np.empty((max(m - 1, 0), 4), np.float64)
        for i in range(max(m - 1, 0)):
            a, c = int(merges[b, i, 0]), int(merges[b, i, 1])
            size[a] += size[c]
            Z[i] = (ident[a], ident[c], 1.0 - float(heights[b, i]), size[a])
            ident[a] = m + i
        out.append(Z)
    return out
