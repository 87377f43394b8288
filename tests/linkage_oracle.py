"""NumPy restatement of hdgnn_hunk_linkage and hdgnn_linkage_cut (include/hdgnn.h), beside the one of hdgnn_hunk_clusters in
oracle/hunk_clusters.py: the same merge loop written again without a threshold, recording (a, c, mean) of every merge, and
the cut of such a record.  It shares only the similarity w with hunk_clusters_one, so the tests compare two independent
formulations of the clustering with each other.

Test infrastructure: not used by the package."""
from __future__ import annotations

import numpy as np

from oracle.hunk_clusters import similarity


def hunk_linkage_one(p1: np.ndarray, n: int, m: int):
    """The merge loop of hunk_clusters_one without a threshold, recording every merge (hdgnn_hunk_linkage): it runs while a
    pair with a non-NaN mean is left (+-inf means merge like any other).  One commit -> (merges (n-1, 2) int32 rows (a, c),
    heights (n-1,) float32, nmerges int); rows from nmerges on are (-1, -1) and NaN; nmerges -1 when m is outside [0, n]."""
    merges = np.full((n - 1, 2), -1, np.int32)
    heights = np.full(n - 1, np.nan, np.float32)
    if m < 0 or m > n:
        return merges, heights, -1
    S = similarity(p1, n, m)
    size = np.ones(m, np.int64)
    # M[i, j] (i < j) = mean(i, j), meaningful where V: both live and the mean is not NaN
    M = np.zeros((m, m), np.float32)
    V = np.zeros((m, m), bool)
    iu = np.triu_indices(m, 1)
    M[iu] = S[iu]
    V[iu] = ~np.isnan(S[iu])
    k = 0
    while V.any():
        best = M[V].max()
        a, c = divmod(int(np.flatnonzero(V & (M == best))[0]), m)     # the smallest (i, j) among equal means (-0 == +0)
        merges[k] = a, c
        heights[k] = M[a, c] + np.float32(0)                            # -0 -> +0
        S[a, :] = S[a, :] + S[c, :]
        S[:, a] = S[a, :]
        size[a] += size[c]
        size[c] = 0
        V[c, :] = V[:, c] = False
        live = np.flatnonzero(size)
        live = live[live != a]
        mean = S[a, live] / (size[a] * size[live]).astype(np.float32)
        lo, hi = np.minimum(live, a), np.maximum(live, a)
        M[lo, hi] = mean
        V[lo, hi] = ~np.isnan(mean)
        k += 1
    return merges, heights, k


def hunk_linkage(probs: np.ndarray, nh=None):
    """probs (B, 2, n(n-1)) float32, nh (B,) or None -> (merges (B, n-1, 2) int32, heights (B, n-1) float32, nmerges (B,) int32)."""
    probs = np.asarray(probs, dtype=np.float32)
    B, _, ncr = probs.shape
    n = (1 + int(round((1 + 4 * ncr) ** 0.5))) // 2
    assert n * (n - 1) == ncr
    merges = np.empty((B, n - 1, 2), np.int32)
    heights = np.empty((B, n - 1), np.float32)
    nmerges = np.empty(B, np.int32)
    for b in range(B):
        merges[b], heights[b], nmerges[b] = hunk_linkage_one(probs[b, 1], n, n if nh is None else int(nh[b]))
    return merges, heights, nmerges


def linkage_cut_one(merges: np.ndarray, heights: np.ndarray, nmerges: int, n: int, m: int, threshold=None, target=None):
    """One commit's record -> (groups (n,) int32, ngroups int) after its first c merges (hdgnn_linkage_cut): c = the longest
    prefix of heights > threshold, or min(nmerges, max(0, m - max(target, 1))).  An inconsistent record gives -1 throughout."""
    bad = np.full(n, -1, np.int32), -1
    if m < 0 or m > n or nmerges < 0 or nmerges > max(m - 1, 0):
        return bad
    absorbed = np.zeros(m, bool)
    for a, c in merges[:nmerges]:
        if not (0 <= a < c < m) or absorbed[a] or absorbed[c]:
            return bad
        absorbed[c] = True
    if target is None:
        above = np.asarray(heights[:nmerges], np.float32) > np.float32(threshold)
        c = int(nmerges if above.all() else np.argmin(above))
    else:
        c = min(int(nmerges), max(0, m - max(int(target), 1)))
    lab = np.arange(n, dtype=np.int32)
    for a, cc in merges[:c]:
        lab[lab == cc] = a
    return lab, n - c


def linkage_cut(merges, heights, nmerges, nh=None, thresholds=None, target=None):
    """(B, n-1, 2), (B, n-1), (B,) records -> (groups (K, B, n) int32, ngroups (K, B) int32) at each threshold, or at target (B,)."""
    B, n = merges.shape[0], merges.shape[1] + 1
    cuts = [dict(threshold=t) for t in thresholds] if target is None else [None]
    groups = np.empty((len(cuts), B, n), np.int32)
    ngroups = np.empty((len(cuts), B), np.int32)
    for k, cut in enumerate(cuts):
        for b in range(B):
            m = n if nh is None else int(nh[b])
            arg = cut if cut is not None else dict(target=target[b])
            groups[k, b], ngroups[k, b] = linkage_cut_one(merges[b], heights[b], int(nmerges[b]), n, m, **arg)
    return groups, ngroups
