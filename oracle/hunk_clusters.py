"""NumPy fp32 restatement of hdgnn_hunk_clusters (include/hdgnn.h): average-linkage (UPGMA) clustering of one commit's real
hunks from the relation probabilities, reproducing the device's merge sequence and every fp32 rounding.

    w(s,t)     = fmax(p1(s,t), p1(t,s))                      s != t < m (NaN only when both are NaN)
    S(A,C)     = sum of w over A x C, kept per pair of live clusters; S(A u B, C) = S(A,C) + S(B,C), one fp32 add
    mean(A,C)  = S(A,C) / float32(|A| |C|)                   IEEE fp32 division
    merge the pair with the largest mean (NaN never), ties to the smaller (min representative, max representative), while
    that mean is > threshold; the merged cluster keeps the smaller representative (its smallest hunk).

Test infrastructure: not used by the package."""
from __future__ import annotations

import numpy as np


def pair_index(n: int) -> np.ndarray:
    """(n, n) int64: p(s,t) = s(n-1) + t - [t > s] for s != t, -1 on the diagonal."""
    s, t = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    p = s * (n - 1) + t - (t > s)
    p[s == t] = -1
    return p


def similarity(p1: np.ndarray, n: int, m: int) -> np.ndarray:
    """(m, m) float32 w of the real hunks from channel 1 (n(n-1),) of one commit; the diagonal is NaN (never used)."""
    p1 = np.asarray(p1, dtype=np.float32)
    idx = pair_index(n)[:m, :m]
    P = np.where(idx >= 0, p1[np.maximum(idx, 0)], np.float32(np.nan)).astype(np.float32)
    return np.fmax(P, P.T)


def hunk_clusters_one(p1: np.ndarray, n: int, m: int, threshold: float):
    """One commit: channel 1 (n(n-1),) float32, m real hunks -> (groups (n,) int32, ngroups int)."""
    if m < 0 or m > n:
        return np.full(n, -1, np.int32), -1
    thr = np.float32(threshold)
    S = similarity(p1, n, m)
    size = np.ones(m, np.int64)
    lab = np.arange(m)
    # M[i, j] (i < j, both live) = mean(i, j); -inf elsewhere and for NaN means: a -inf mean can never be > threshold, so
    # treating "no pair" and NaN as -inf stops exactly where the specification stops
    M = np.full((m, m), -np.inf, np.float32)
    iu = np.triu_indices(m, 1)
    M[iu] = S[iu]
    M[np.isnan(M)] = -np.inf
    merges = 0
    while m - merges > 1:
        k = int(np.argmax(M))                     # first maximum in row-major order = the smallest (i, j) among equal means
        a, c = divmod(k, m)
        if not (M[a, c] > thr):
            break
        S[a, :] = S[a, :] + S[c, :]
        S[:, a] = S[a, :]
        size[a] += size[c]
        size[c] = 0
        lab[lab == c] = a
        M[c, :] = -np.inf
        M[:, c] = -np.inf
        live = np.flatnonzero(size)
        live = live[live != a]
        mean = S[a, live] / (size[a] * size[live]).astype(np.float32)
        mean[np.isnan(mean)] = -np.inf
        lo, hi = np.minimum(live, a), np.maximum(live, a)
        M[lo, hi] = mean
        merges += 1
    groups = np.arange(n, dtype=np.int32)
    groups[:m] = lab
    return groups, n - merges


def hunk_clusters(probs: np.ndarray, nh=None, threshold: float = 0.5):
    """probs (B, 2, n(n-1)) float32, nh (B,) or None -> (groups (B, n) int32, ngroups (B,) int32)."""
    probs = np.asarray(probs, dtype=np.float32)
    B, _, ncr = probs.shape
    n = (1 + int(round((1 + 4 * ncr) ** 0.5))) // 2
    assert n * (n - 1) == ncr
    groups = np.empty((B, n), np.int32)
    ngroups = np.empty(B, np.int32)
    for b in range(B):
        m = n if nh is None else int(nh[b])
        groups[b], ngroups[b] = hunk_clusters_one(probs[b, 1], n, m, threshold)
    return groups, ngroups
