"""Loader for the reference's on-disk commit data, producing the compact wire format of the hot path.

Reads exactly what utils2.py:22-27 reads (paths relative to `root`, default the CWD):

    ./Adjset/{repo}/Cutting_Adjs/CAdjs_{step}.npy          (N, Ne, Ne)  entity adjacency, diagonal = node attribute
    ./Adjset/{repo}/Cutting_Adjs/CHunkAdjs_{step}.npy      (N, Nc, Nc)  hunk adjacency (= label)
    ./dataset/{repo}/IndexPathList/IndexPathList_{step}.pkl  joblib list of N text-file paths (one hunk key per entity line)
    ./dataset/{repo}/HunkIDdict/HunkIDmap_{step}.pkl         joblib list of N dicts  key -> hunk number

and keeps the index semantics of utils2.py:29-47 and :111-137 (diagonal -> x, 'null' lines, the Nc cut,
the first-Ne-lines cut), but stores them as (adj u8, x f32, hmap i32, L i32, Y u8) instead of the
dense one-hot tensors Es/Et/Cs/Ct/Esc/Etc (90.8 MB per commit at glide).  `read_data(self, step)`
keeps the reference's 12-tuple for small problems (tests / migration); `read_compact` is what
graph2graph.train/test use.
"""
from __future__ import annotations

import os
from typing import Tuple

import numpy as np

from .synthetic import CommitBatch

NULL_KEY = "null"


def _paths(root, repo, step):
    return (os.path.join(root, "Adjset", repo, "Cutting_Adjs", f"CAdjs_{step}.npy"),
            os.path.join(root, "Adjset", repo, "Cutting_Adjs", f"CHunkAdjs_{step}.npy"),
            os.path.join(root, "dataset", repo, "IndexPathList", f"IndexPathList_{step}.pkl"),
            os.path.join(root, "dataset", repo, "HunkIDdict", f"HunkIDmap_{step}.pkl"))


def _cache_path(root, repo, step, Ne, Nc):
    return os.path.join(root, "Intermediate_products", repo, f"compact_{step}_{Ne}_{Nc}.npz")


def _grids_host(x_raw, y_raw, Ne, Nc):
    """Array half of the loader on the host (NumPy): the checker of the device loader and the form the CPU tests use."""
    ie, ic = np.arange(Ne), np.arange(Nc)
    x = x_raw[:, ie, ie].astype(np.float32)                      # utils2.py:31-36: node attribute = diagonal
    adj_f = np.array(x_raw, dtype=np.float64, copy=True)
    adj_f[:, ie, ie] = 0                                          # utils2.py:46
    y_f = np.array(y_raw, dtype=np.float64, copy=True)
    y_f[:, ic, ic] = 0                                            # utils2.py:47
    # utils2.py:82,105 index a size-2 axis with int(value): anything but 0/1 is an IndexError there
    for name, arr in (("CAdjs", adj_f), ("CHunkAdjs", y_f)):
        if not np.isfinite(arr).all():
            raise IndexError(f"{name}: off-diagonal entries must truncate to 0 or 1 (utils2.py:82,105)")
        iv = arr.astype(np.int64)                                 # int() truncates toward zero
        if iv.min() < -2 or iv.max() > 1:
            raise IndexError(f"{name}: off-diagonal entries must truncate to 0 or 1 (utils2.py:82,105)")
    adj = (adj_f.astype(np.int64) % 2).astype(np.uint8)           # int(v) in {-2,-1,0,1}; python index -1 == 1, -2 == 0
    Y = (y_f.astype(np.int64) % 2).astype(np.uint8)
    return adj, x, Y


def _grids_device(x_raw, y_raw, Ne, Nc, device):
    """Array half of the loader on the GPU (hdgnn_compact_from_raw, csrc/k_io.cu); raises IndexError like the host form."""
    import torch
    from .engine import compact_from_raw_device
    adj, x = compact_from_raw_device(torch.as_tensor(np.ascontiguousarray(x_raw)).to(device))
    Y, _ = compact_from_raw_device(torch.as_tensor(np.ascontiguousarray(y_raw)).to(device), want_diag=False)
    return adj[:, :, :Ne].cpu().numpy(), x.cpu().numpy(), Y[:, :, :Nc].cpu().numpy()


def _index_maps(index_lines, hunk_maps, N, Ne, Nc):
    """String half of the loader (utils2.py:111-137): per commit the hunk number of every index line."""
    hmap = np.full((N, Ne), -1, dtype=np.int32)
    L = np.zeros(N, dtype=np.int32)
    for b in range(N):
        lines = list(index_lines[b])[:Ne]                         # utils2.py:121
        L[b] = len(lines)
        m = hunk_maps[b]
        for i, line in enumerate(lines):
            key = line.strip()
            if key != NULL_KEY:                                   # utils2.py:128-132
                num = int(m[key])
                if num < Nc:
                    hmap[b, i] = num if num >= 0 else num + Nc    # a negative number indexes from the end in numpy
    return hmap, L


def compact_from_raw(x_raw, y_raw, index_lines, hunk_maps, Ne, Nc, device=None) -> CommitBatch:
    """x_raw (N,Ne,Ne), y_raw (N,Nc,Nc): arrays as stored; index_lines: per commit the list of lines of
    its IndexPath file; hunk_maps: per commit dict key -> number.  device: CUDA device -> the array half runs on
    the GPU (what graph2graph uses); None -> NumPy (CPU tests, the checker).
    The number of real hunks of commit b is taken as nh[b] = min(Nc, len(hunk_maps[b])).  This assumes that the hunk numbers
    0 .. len-1 of a commit's map occupy rows 0 .. len-1 of its CHunkAdjs grid and that the rest is padding, which is what
    write_dataset writes; it has not been verified against the reference's data blob, which is missing."""
    x_raw = np.asarray(x_raw)
    y_raw = np.asarray(y_raw)
    N = x_raw.shape[0]
    if x_raw.shape[1:] != (Ne, Ne) or y_raw.shape != (N, Nc, Nc):
        raise ValueError(f"adjacency shapes {x_raw.shape} / {y_raw.shape} do not match Ne={Ne}, Nc={Nc}")
    adj, x, Y = _grids_host(x_raw, y_raw, Ne, Nc) if device is None else _grids_device(x_raw, y_raw, Ne, Nc, device)
    hmap, L = _index_maps(index_lines, hunk_maps, N, Ne, Nc)
    nh = np.array([min(Nc, len(m)) for m in hunk_maps], dtype=np.int32)
    return CommitBatch(adj, x, hmap, L, Y, nh)


def read_compact(repo: str, step: int, Ne: int, Nc: int, root: str = ".", cache: bool = True, device=None) -> CommitBatch:
    """compact_from_raw of the files of utils2.py:22-25, through the cache Intermediate_products/{repo}/compact_*.npz.  A cache
    written before the hunk counts were stored loads with nh = None (every Nc hunk counts as real)."""
    cp = _cache_path(root, repo, step, Ne, Nc)
    if cache and os.path.exists(cp):
        z = np.load(cp)
        return CommitBatch(z["adj"], z["x"], z["hmap"], z["L"], z["Y"], z["nh"] if "nh" in z.files else None)
    import joblib
    pa, py, pi, ph = _paths(root, repo, step)
    for p in (pa, py, pi, ph):
        if not os.path.exists(p):
            raise FileNotFoundError(f"{p} (expected by utils2.py:22-25 relative to the working directory)")
    x_raw = np.load(pa, allow_pickle=True)
    y_raw = np.load(py, allow_pickle=True)
    with open(pi, "rb") as f:
        index_paths = joblib.load(f)
    with open(ph, "rb") as f:
        hunk_maps = joblib.load(f)
    lines = []
    for p in index_paths:
        q = p if os.path.isabs(p) or os.path.exists(p) else os.path.join(root, p)
        with open(q) as f:
            lines.append(f.readlines())
    cb = compact_from_raw(x_raw, y_raw, lines, hunk_maps, Ne, Nc, device=device)
    if cache and int(os.environ.get("RANK", "0")) == 0:
        # one writer (rank 0), temporary file + atomic rename: a rank arriving later never sees a half-written zip
        os.makedirs(os.path.dirname(cp), exist_ok=True)          # the reference needs this dir to pre-exist (Q14)
        tmp = f"{cp}.{os.getpid()}.tmp.npz"
        np.savez_compressed(tmp, adj=cb.adj, x=cb.x, hmap=cb.hmap, L=cb.L, Y=cb.Y, nh=cb.nh)
        os.replace(tmp, cp)
    return cb


def split_half(cb: CommitBatch) -> Tuple[CommitBatch, CommitBatch]:
    """First half train / second half test (utils2.py:140-149)."""
    h = int(cb.B / 2)
    return cb.slice(0, h), cb.slice(h, cb.B)


def pair_index(n: int):
    """Row-major ordered pairs (i, j), i != j: p = i (n-1) + j - [j > i] (utils2.py:69-83)."""
    i, j = np.divmod(np.arange(n * n), n)
    keep = i != j
    return i[keep], j[keep]


def edge_onehot(lab: np.ndarray) -> np.ndarray:
    """(N,n,n) {0,1} -> (N,2,n(n-1)) float32 one-hot over pairs; channel int(value) (utils2.py:82,105)."""
    n = lab.shape[1]
    i, j = pair_index(n)
    v = lab[:, i, j].astype(np.float32)
    return np.stack([1.0 - v, v], 1)


def dense_feeds(cb: CommitBatch, Ne: int, Nc: int, lead: int = None):
    """The dense arrays of utils2.py:50-137 from a compact batch (vectorised).  `lead` = leading
    dimension of Es/Et/Cs/Ct/Esc/Etc (the reference hard-codes 100, utils2.py:50-61)."""
    N = cb.B
    lead = N if lead is None else lead
    Ner, Ncr = Ne * (Ne - 1), Nc * (Nc - 1)
    ei, ej = pair_index(Ne)
    ci, cj = pair_index(Nc)
    Es = np.zeros((lead, Ne, Ner), np.float32); Et = np.zeros((lead, Ne, Ner), np.float32)
    Es[:, ei, np.arange(Ner)] = 1; Et[:, ej, np.arange(Ner)] = 1
    Cs = np.zeros((lead, Nc, Ncr), np.float32); Ct = np.zeros((lead, Nc, Ncr), np.float32)
    Cs[:, ci, np.arange(Ncr)] = 1; Ct[:, cj, np.arange(Ncr)] = 1
    E_edge = np.zeros((lead, 2, Ner), np.float32); C_edge = np.zeros((lead, 2, Ncr), np.float32)
    E_edge[:N] = edge_onehot(cb.adj); C_edge[:N] = edge_onehot(cb.Y)
    Esc = np.zeros((lead, Nc, Ner), np.float32); Etc = np.zeros((lead, Nc, Ner), np.float32)
    for b in range(N):
        Lb = int(cb.L[b])
        li, lj = pair_index(Lb)
        q = np.arange(Lb * (Lb - 1))                              # local counter cnt2 (utils2.py:123-137)
        hs, ht = cb.hmap[b, li], cb.hmap[b, lj]
        Esc[b, hs[hs >= 0], q[hs >= 0]] = 1
        Etc[b, ht[ht >= 0], q[ht >= 0]] = 1
    node = cb.x.astype(np.float64).reshape(N, 1, Ne)
    return node, E_edge, C_edge, Es, Et, Cs, Ct, Esc, Etc


def read_data(self, step, root: str = ".", max_bytes: float = 8e9):
    """Drop-in for utils2.read_data(self, step): the 12-tuple of dense arrays
    (E_node_train, E_node_test, E_edge_train, E_edge_test, C_edge_train, C_edge_test, Es_data, Et_data,
    Cs_label, Ct_label, Esc_data, Etc_data), utils2.py:248-253.  Refuses problems whose one-hot tensors
    would not fit in `max_bytes` (the reference needs 9 GB at glide); the hot path never calls this."""
    cb = read_compact(self.Repo, step, self.Ne, self.Nc, root=root)
    Ner, Ncr = self.Ne * (self.Ne - 1), self.Nc * (self.Nc - 1)
    need = 4.0 * cb.B * (2 * self.Ne * Ner + 2 * self.Nc * Ncr + 2 * self.Nc * Ner)
    if need > max_bytes:
        raise MemoryError(f"dense one-hot feeds need {need / 1e9:.1f} GB; use read_compact (the hot path does)")
    node, E_edge, C_edge, Es, Et, Cs, Ct, Esc, Etc = dense_feeds(cb, self.Ne, self.Nc)
    h = int(cb.B / 2)
    return (node[:h], node[h:], E_edge[:h], E_edge[h:], C_edge[:h], C_edge[h:], Es, Et, Cs, Ct, Esc, Etc)


def write_dataset(cb: CommitBatch, repo: str, step: int, root: str = ".", hunk_key=lambda b, c: f"hunk_{b}_{c}"):
    """Write a compact batch in the reference's on-disk formats (synthetic stand-in for the missing
    Adjset/glide.zip): the diagonal carries x, entity lines map to hunk keys / 'null', lines beyond L
    are simply absent."""
    import joblib
    pa, py, pi, ph = _paths(root, repo, step)
    for p in (pa, py, pi, ph):
        os.makedirs(os.path.dirname(p), exist_ok=True)
    N, Ne, Nc = cb.B, cb.Ne, cb.Nc
    xa = cb.adj.astype(np.float64)
    xa[:, np.arange(Ne), np.arange(Ne)] = cb.x
    np.save(pa, xa)
    np.save(py, cb.Y.astype(np.float64))
    idx_dir = os.path.join(root, "dataset", repo, "IndexPath", str(step))
    os.makedirs(idx_dir, exist_ok=True)
    paths, maps = [], []
    for b in range(N):
        m = {hunk_key(b, c): c for c in range(Nc + 4)}            # ids >= Nc exist in the map and are cut (utils2.py:131)
        p = os.path.join(idx_dir, f"index_{b}.txt")
        with open(p, "w") as f:
            for i in range(int(cb.L[b])):
                hc = int(cb.hmap[b, i])
                f.write((NULL_KEY if hc < 0 else hunk_key(b, hc)) + "\n")
        paths.append(p); maps.append(m)
    with open(pi, "wb") as f:
        joblib.dump(paths, f)
    with open(ph, "wb") as f:
        joblib.dump(maps, f)
