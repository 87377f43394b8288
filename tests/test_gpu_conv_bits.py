"""The legacy operator (model.py:335-403) fed label bitmaps (HDGNN_P_LABEL_BITS) instead of byte grids: normalize_propagate,
map_conv and both backwards.  Where both formats run the same kernel the results are bitwise equal to the byte-grid call;
where the kernel selection may differ, and beyond the byte grid's size limit, they match the fp64 oracle."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import hdgnn_oracle as O

gpu = pytest.mark.gpu
P_FORCED = 8 | 16               # P_NO_TENSOR | P_TENSOR_V1: the same forced kernel for both formats


def _adj(B, N, p, seed):
    rng = np.random.default_rng(seed)
    a = (rng.random((B, N, N)) < p).astype(np.uint8)
    a[:, np.arange(N), np.arange(N)] = 0
    return a


def _formats(adj):
    """(B,N,N) uint8 numpy -> (byte grid, label bitmap packed on the device (int32)), both CUDA."""
    from hdgnn_b200.engine import _pitched, pack_label_bits_device
    grid = _pitched(torch.tensor(adj).cuda())
    return grid, pack_label_bits_device(grid)


def _dirty(bits, N):
    """The same bitmap with every diagonal bit and every padding bit (columns >= N) set."""
    b = bits.cpu().numpy().view(np.uint32).copy()
    wp = b.shape[2]
    col = np.arange(wp * 32)
    pad = np.packbits((col >= N).astype(np.uint8), bitorder="little").view("<u4")
    b |= pad[None, None, :]
    i = np.arange(N)
    b[:, i, i >> 5] |= (np.uint32(1) << (i & 31).astype(np.uint32))
    return torch.from_numpy(b.view(np.int32)).cuda()


def _ref_propagate(adj, H, W, bias, eps, self_loop, relu, transpose):
    A = adj.astype(np.float64)
    N = A.shape[1]
    if self_loop:
        A = A + np.eye(N)
    d = (A.sum(2) + eps) ** -0.5
    M = np.transpose(A, (0, 2, 1)) if transpose else A
    Ahat = d[:, :, None] * M * d[:, None, :]
    Z = H.astype(np.float64) if W is None else H.astype(np.float64) @ W.astype(np.float64)
    out = Ahat @ Z + (0 if bias is None else bias.astype(np.float64))
    return (np.maximum(out, 0) if relu else out), d


def _autograd_propagate(adj, H, W, bias, dOut, flags):
    A = torch.tensor(adj, dtype=torch.float64)
    N = A.shape[1]
    if flags & 1:
        A = A + torch.eye(N, dtype=torch.float64)
    d = (A.sum(2) + float(np.float32(1e-3))) ** -0.5
    M = A if flags & 4 else A.transpose(1, 2)
    Ahat = d[:, :, None] * M * d[:, None, :]
    Ht = torch.tensor(H, requires_grad=True); Wt = torch.tensor(W, requires_grad=True); bt = torch.tensor(bias, requires_grad=True)
    pre = Ahat @ (Ht @ Wt) + bt
    out_ref = torch.relu(pre) if flags & 2 else pre
    return torch.autograd.grad((out_ref * torch.tensor(dOut)).sum(), [Ht, Wt, bt])


def _autograd_map_conv(adj, x, flags):
    N = adj.shape[1]
    th = torch.tensor([0.13, -0.21], dtype=torch.float64, requires_grad=True)
    xt = torch.tensor(x, requires_grad=True)
    A = torch.tensor(adj, dtype=torch.float64)
    if flags & 1:
        A = A + torch.eye(N, dtype=torch.float64)
    d = (A.sum(2) + float(np.float32(1e-3))) ** -0.5
    Ahat = d[:, :, None] * (A if flags & 4 else A.transpose(1, 2)) * d[:, None, :]
    t = torch.softmax(th, 0)
    Lx = (2.0 / 1.5) * (xt - (Ahat @ xt[..., None])[..., 0]) - xt
    loss = (((xt * (t[0] * xt + t[1] * Lx)).sum(1)) ** 2).mean()
    gx, gt = torch.autograd.grad(loss, [xt, th])
    return th.detach(), gx, gt


def _rel(a, r):
    a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
    r = r.numpy() if isinstance(r, torch.Tensor) else r
    return float(np.abs(a - r).max() / max(np.abs(r).max(), 1e-30))


def _same(x, y):
    return all(torch.equal(a, b) for a, b in zip(x, y) if a is not None or b is not None)


# ---- same kernel, same bits ----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("B,N,d_in,d_out,p", [(3, 9, 4, 4, 0.3), (4, 50, 7, 20, 0.1), (2, 200, 20, 20, 0.05), (2, 250, 1, 1, 0.05),
                                              (1, 300, 20, 32, 0.02)])
@pytest.mark.parametrize("flags", [0, 1, 2 | 4, 1 | 2, 8, 8 | 1 | 2 | 4, 16, 16 | 1 | 4])
def test_normalize_propagate_bits_equal_bytes(B, N, d_in, d_out, p, flags):
    from hdgnn_b200.engine import normalize_propagate
    rng = np.random.default_rng(N + flags)
    adj = _adj(B, N, p, N)
    H = rng.normal(size=(B, N, d_in)).astype(np.float32)
    W = None if d_in == d_out and flags in (0, 8) else rng.normal(scale=0.3, size=(d_in, d_out)).astype(np.float32)
    bias = rng.normal(size=d_out).astype(np.float32) if flags & 2 else None
    grid, bits = _formats(adj)
    Hd, Wd = torch.tensor(H).cuda(), None if W is None else torch.tensor(W).cuda()
    bd = None if bias is None else torch.tensor(bias).cuda()
    out_b, dinv_b = normalize_propagate(bits, Hd, Wd, bd, eps=1e-3, flags=flags)
    torch.cuda.synchronize()
    if flags & P_FORCED or N <= 200:
        out_g, dinv_g = normalize_propagate(grid, Hd, Wd, bd, eps=1e-3, flags=flags)
        torch.cuda.synchronize()
        assert torch.equal(out_b, out_g) and torch.equal(dinv_b, dinv_g)
    else:           # the persistent kernel may take the bitmap where the byte grid runs another kernel
        ref, d = _ref_propagate(adj, H, W, bias, 1e-3, bool(flags & 1), bool(flags & 2), not (flags & 4))
        assert _rel(dinv_b, d) < 1e-6
        assert _rel(out_b, ref) < 1e-5


@gpu
@pytest.mark.parametrize("B,N,d_in,d_out,p", [(3, 9, 4, 4, 0.3), (4, 50, 7, 20, 0.1), (2, 200, 20, 20, 0.05), (2, 300, 20, 32, 0.02)])
@pytest.mark.parametrize("flags", [0, 2, 1 | 2, 4, 8 | 2, 16])
def test_normalize_propagate_backward_bits_equal_bytes(B, N, d_in, d_out, p, flags):
    from hdgnn_b200.engine import normalize_propagate, normalize_propagate_backward
    rng = np.random.default_rng(N + 3 * flags)
    adj = _adj(B, N, p, N + 5)
    H = rng.normal(size=(B, N, d_in))
    W = rng.normal(scale=0.3, size=(d_in, d_out))
    bias = rng.normal(size=d_out) if flags & 2 else np.zeros(d_out)
    dOut = rng.normal(size=(B, N, d_out))
    grid, bits = _formats(adj)
    Hd, Wd = torch.tensor(H, dtype=torch.float32).cuda(), torch.tensor(W, dtype=torch.float32).cuda()
    bd = torch.tensor(bias, dtype=torch.float32).cuda() if flags & 2 else None
    dOd = torch.tensor(dOut, dtype=torch.float32).cuda()
    out_b, _ = normalize_propagate(bits, Hd, Wd, bd, eps=1e-3, flags=flags)
    got = normalize_propagate_backward(bits, Hd, dOd, W=Wd, out=out_b, eps=1e-3, flags=flags)
    torch.cuda.synchronize()
    if flags & P_FORCED or N <= 200:
        out_g, _ = normalize_propagate(grid, Hd, Wd, bd, eps=1e-3, flags=flags)
        want = normalize_propagate_backward(grid, Hd, dOd, W=Wd, out=out_g, eps=1e-3, flags=flags)
        torch.cuda.synchronize()
        assert torch.equal(out_b, out_g) and _same(got, want)
    else:
        gH, gW, gb = _autograd_propagate(adj, H, W, bias, dOut, flags)
        assert _rel(got[0], gH) < 2e-5 and _rel(got[1], gW) < 2e-5 and _rel(got[2], gb) < 2e-5


@gpu
@pytest.mark.parametrize("B,N,p", [(3, 6, 0.4), (5, 40, 0.15), (4, 200, 0.05), (2, 333, 0.03)])
@pytest.mark.parametrize("flags", [0, 1, 4, 1 | 4, 16])
def test_map_conv_bits_equal_bytes(B, N, p, flags):
    from hdgnn_b200.engine import map_conv
    rng = np.random.default_rng(N)
    adj = _adj(B, N, p, N + 1)
    x = torch.tensor(rng.integers(0, 10, size=(B, N)).astype(np.float32) / 3.0).cuda()
    theta = torch.tensor([0.13, -0.21]).cuda()
    grid, bits = _formats(adj)
    got = map_conv(bits, x, theta, flags=flags)
    want = map_conv(grid, x, theta, flags=flags)
    torch.cuda.synchronize()
    assert _same(got, want)


@gpu
@pytest.mark.parametrize("B,N,p", [(3, 6, 0.4), (4, 200, 0.05), (2, 333, 0.03)])
@pytest.mark.parametrize("flags", [0, 1, 4, 1 | 4])
def test_map_conv_backward_bits_equal_bytes(B, N, p, flags):
    from hdgnn_b200.engine import map_conv_backward
    rng = np.random.default_rng(N + flags)
    adj = _adj(B, N, p, N + 2)
    x = torch.tensor(rng.integers(0, 10, size=(B, N)).astype(np.float32) / 3.0).cuda()
    theta = torch.tensor([0.13, -0.21]).cuda()
    grid, bits = _formats(adj)
    got = map_conv_backward(bits, x, theta, flags=flags, gscale=0.7)
    want = map_conv_backward(grid, x, theta, flags=flags, gscale=0.7)
    torch.cuda.synchronize()
    assert _same(got, want)


@gpu
@pytest.mark.parametrize("flags", [0, 4, 1 | 2])
def test_normalize_propagate_bits_persistent_many_commits(flags):
    """More commits than SMs: every CTA of the persistent tcgen05 kernel walks several bitmap tiles with the prefetch."""
    from hdgnn_b200.engine import normalize_propagate
    B, N, d = 450, 200, 20
    rng = np.random.default_rng(3)
    adj = _adj(B, N, 0.05, 9)
    H = torch.tensor(rng.normal(size=(B, N, d)).astype(np.float32)).cuda()
    bias = torch.tensor(rng.normal(size=d).astype(np.float32)).cuda() if flags & 2 else None
    grid, bits = _formats(adj)
    got = normalize_propagate(bits, H, None, bias, eps=1e-3, flags=flags)
    want = normalize_propagate(grid, H, None, bias, eps=1e-3, flags=flags)
    torch.cuda.synchronize()
    assert _same(got, want)


# ---- the diagonal and the padding bits are ignored -----------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("N", [50, 200, 400])
def test_diagonal_and_padding_bits_are_ignored(N):
    from hdgnn_b200.engine import map_conv, map_conv_backward, normalize_propagate, normalize_propagate_backward
    B, d = 3, 20
    rng = np.random.default_rng(N)
    adj = _adj(B, N, 0.1, N + 7)
    _, clean = _formats(adj)
    dirty = _dirty(clean, N)
    assert not torch.equal(clean, dirty)
    H = torch.tensor(rng.normal(size=(B, N, d)).astype(np.float32)).cuda()
    W = torch.tensor(rng.normal(scale=0.3, size=(d, d)).astype(np.float32)).cuda()
    dOut = torch.tensor(rng.normal(size=(B, N, d)).astype(np.float32)).cuda()
    x = torch.tensor(rng.normal(size=(B, N)).astype(np.float32)).cuda()
    theta = torch.tensor([0.13, -0.21]).cuda()
    for flags in (0, 4, 8, 16, 1 | 2):
        outs = [normalize_propagate(a, H, W, eps=1e-3, flags=flags) for a in (clean, dirty)]
        assert _same(*outs), flags
    for flags in (0, 1 | 2):
        out, _ = normalize_propagate(clean, H, W, eps=1e-3, flags=flags)
        grads = [normalize_propagate_backward(a, H, dOut, W=W, out=out, eps=1e-3, flags=flags) for a in (clean, dirty)]
        assert _same(*grads), flags
    for flags in (0, 1, 1 | 4):
        assert _same(*[map_conv(a, x, theta, flags=flags) for a in (clean, dirty)]), flags
        assert _same(*[map_conv_backward(a, x, theta, flags=flags) for a in (clean, dirty)]), flags
    torch.cuda.synchronize()


# ---- beyond the byte grid's limit ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("N,d", [(400, 20), (512, 32)])
def test_bits_beyond_the_byte_grid_limit(N, d):
    """A bitmap tile is 1/8 of a byte tile: every entry point runs up to N = 512, where a byte grid no longer fits one SM."""
    from hdgnn_b200.engine import map_conv, map_conv_backward, normalize_propagate, normalize_propagate_backward
    B, p = 2, 0.03
    rng = np.random.default_rng(N)
    adj = _adj(B, N, p, N + 11)
    _, bits = _formats(adj)
    H = rng.normal(size=(B, N, d))
    W = rng.normal(scale=0.3, size=(d, d))
    Hd, Wd = torch.tensor(H, dtype=torch.float32).cuda(), torch.tensor(W, dtype=torch.float32).cuda()
    for flags in (0, 1 | 2 | 4):
        bias = rng.normal(size=d) if flags & 2 else np.zeros(d)
        bd = torch.tensor(bias, dtype=torch.float32).cuda()
        out, dinv = normalize_propagate(bits, Hd, Wd, bd, eps=1e-3, flags=flags)
        torch.cuda.synchronize()
        ref, dd = _ref_propagate(adj, H.astype(np.float32), W.astype(np.float32), bias.astype(np.float32), 1e-3,
                                 bool(flags & 1), bool(flags & 2), not (flags & 4))
        assert _rel(dinv, dd) < 1e-6 and _rel(out, ref) < 1e-5, flags
        dOut = rng.normal(size=(B, N, d))
        dH, dW, db = normalize_propagate_backward(bits, Hd, torch.tensor(dOut, dtype=torch.float32).cuda(), W=Wd, out=out,
                                                  eps=1e-3, flags=flags)
        torch.cuda.synchronize()
        gH, gW, gb = _autograd_propagate(adj, H, W, bias, dOut, flags)
        assert _rel(dH, gH) < 2e-5 and _rel(dW, gW) < 2e-5 and _rel(db, gb) < 2e-5, flags
    x = rng.integers(0, 10, size=(B, N)).astype(np.float64) / 3.0
    xd = torch.tensor(x, dtype=torch.float32).cuda()
    theta = torch.tensor([0.13, -0.21], dtype=torch.float64)
    loss, _ = map_conv(bits, xd, theta.float().cuda())
    torch.cuda.synchronize()
    ref = float(O.map_conv_closed(theta, torch.tensor(adj), torch.tensor(x)))
    assert abs(loss.item() - ref) <= 1e-4 * abs(ref)
    for flags in (0, 1 | 4):
        th, gx, gt = _autograd_map_conv(adj, x, flags)
        dx, dth = map_conv_backward(bits, xd, th.float().cuda(), flags=flags, gscale=0.7)
        torch.cuda.synchronize()
        assert _rel(dx, 0.7 * gx) < 5e-5 and _rel(dth, 0.7 * gt) < 5e-5, flags


# ---- the reference's own model.py ------------------------------------------------------------------------------------------
@gpu
def test_bits_match_reference_model_py_golden():
    """tests/golden/legacy_toy.npz (the reference's model.py:335-417 over the shim) packed to label bitmaps on the host."""
    from hdgnn_b200.engine import map_conv, map_conv_backward, normalize_propagate, pack_label_bits
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "legacy_toy.npz"))
    mb, No = z["adj"].shape[:2]
    bits = torch.from_numpy(pack_label_bits(z["adj"])).cuda()
    assert bits.dtype == torch.uint32
    x = torch.tensor(z["O"].reshape(mb, No), dtype=torch.float32).cuda()
    theta = torch.tensor(z["theta"], dtype=torch.float32).cuda()
    loss, _ = map_conv(bits, x, theta)
    torch.cuda.synchronize()
    assert abs(loss.item() - float(z["loss"])) <= 1e-5 * abs(float(z["loss"]))
    Ahat = np.eye(No) - 0.75 * (z["t_k"][:, 1] + np.eye(No))
    H = np.random.default_rng(5).normal(size=(mb, No, 20)).astype(np.float32)
    for flags in (0, 8, 16):
        out, _ = normalize_propagate(bits, torch.tensor(H).cuda(), flags=flags)
        torch.cuda.synchronize()
        ref = Ahat @ H.astype(np.float64)
        assert np.abs(out.cpu().numpy() - ref).max() / np.abs(ref).max() < 1e-5, flags
    dx, dth = map_conv_backward(bits, x, theta)
    torch.cuda.synchronize()
    ref_dx, ref_dth = z["dO"].reshape(mb, No), z["dtheta"]
    assert np.abs(dx.cpu().numpy() - ref_dx).max() / np.abs(ref_dx).max() < 1e-5
    assert np.abs(dth.cpu().numpy() - ref_dth).max() / np.abs(ref_dth).max() < 1e-5


# ---- argument checks -------------------------------------------------------------------------------------------------------
def _c_calls(N, adj_ptr, pitch, flags):
    """The four legacy entry points with fake device pointers: each must refuse the adjacency before any CUDA call."""
    from hdgnn_b200._lib import lib
    f = C.c_void_p(1 << 20)
    return {
        "normalize_propagate": lib.hdgnn_normalize_propagate(2, N, adj_ptr, pitch, f, 20, None, None, 20, 1e-3, flags, f, None, None),
        "map_conv": lib.hdgnn_map_conv(2, N, adj_ptr, pitch, f, f, 1.5, 1e-3, flags, f, None, None),
        "normalize_propagate_backward": lib.hdgnn_normalize_propagate_backward(2, N, adj_ptr, pitch, f, 20, None, 20, 1e-3, flags,
                                                                              None, f, f, None, None, f, None),
        "map_conv_backward": lib.hdgnn_map_conv_backward(2, N, adj_ptr, pitch, f, f, 1.5, 1e-3, flags, 1.0, f, None, None, None),
    }


@pytest.mark.parametrize("N", [9, 200, 512])
def test_bitmap_pitch_and_alignment_are_checked_before_launch(N):
    from hdgnn_b200 import _lib
    from hdgnn_b200.engine import P_LABEL_BITS, bit_words, label_pitch
    aligned, pitch = C.c_void_p(1 << 24), 4 * bit_words(N)
    wrong = {label_pitch(N), pitch + 16, pitch - 16, 4 * ((N + 31) // 32)} - {pitch, 0}     # byte pitch, unpadded rows, ...
    bad = [(aligned, p) for p in sorted(wrong)] + [(C.c_void_p((1 << 24) + 4), pitch)]      # ... and a misaligned base
    for adj, p in bad:
        for name, rc in _c_calls(N, adj, p, P_LABEL_BITS).items():
            assert rc == _lib.E_INVALID, (name, p, adj.value)
    for name, rc in _c_calls(_lib.MAX_N + 1, aligned, 4 * 16, P_LABEL_BITS).items():
        assert rc == _lib.E_INVALID, name


def test_bitmap_arguments_are_checked_in_python():
    from hdgnn_b200.engine import (P_LABEL_BITS, bit_words, map_conv, map_conv_backward, normalize_propagate,
                                   normalize_propagate_backward)
    N = 200
    H, x, theta = torch.zeros(1, N, 20), torch.zeros(1, N), torch.zeros(2)
    calls = [lambda a, f: normalize_propagate(a, H, flags=f), lambda a, f: map_conv(a, x, theta, flags=f),
             lambda a, f: normalize_propagate_backward(a, H, H, flags=f), lambda a, f: map_conv_backward(a, x, theta, flags=f)]
    for fn in calls:
        for dt in (torch.int32, torch.uint32):
            with pytest.raises(ValueError, match="bit_words"):
                fn(torch.zeros(1, N, bit_words(N) - 1, dtype=dt), 0)
        with pytest.raises(ValueError, match="P_LABEL_BITS"):
            fn(torch.zeros(1, N, N, dtype=torch.uint8), P_LABEL_BITS)


@gpu
def test_misaligned_bitmap_is_refused():
    from hdgnn_b200._lib import E_INVALID, HdgnnError
    from hdgnn_b200.engine import bit_words, map_conv, normalize_propagate
    N = 200
    wp = bit_words(N)
    flat = torch.zeros(N * wp + 1, dtype=torch.int32, device="cuda")
    bits = flat[1:].view(1, N, wp)          # contiguous, 4 bytes past a 16-byte boundary
    with pytest.raises(HdgnnError) as e:
        normalize_propagate(bits, torch.zeros(1, N, 20, device="cuda"))
    assert e.value.code == E_INVALID
    with pytest.raises(HdgnnError) as e:
        map_conv(bits, torch.zeros(1, N, device="cuda"), torch.zeros(2, device="cuda"))
    assert e.value.code == E_INVALID
