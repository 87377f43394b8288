"""CPU checks of the average-linkage hunk clusters: the NumPy restatement of their specification (oracle/hunk_clusters.py)
equals scipy's average linkage cut at 1 - threshold and keeps apart two groups that one confident false-positive pair chains
together under connected components."""
import numpy as np
from scipy.cluster.hierarchy import fcluster, linkage
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial.distance import squareform

from oracle.hunk_clusters import hunk_clusters, hunk_clusters_one, pair_index


def _probs_of(P1: np.ndarray) -> np.ndarray:
    """(B, n, n) channel-1 grids -> (B, 2, n(n-1)) float32 in the relation head's pair order, channel 0 = 1 - channel 1."""
    B, n, _ = P1.shape
    idx = pair_index(n)
    off = idx >= 0
    out = np.zeros((B, 2, n * (n - 1)), np.float32)
    out[:, 1][:, idx[off]] = P1[:, off]
    out[:, 0] = 1 - out[:, 1]
    return out


def _smallest_index_labels(lab: np.ndarray) -> np.ndarray:
    first = {}
    for i, v in enumerate(lab):
        first.setdefault(v, i)
    return np.array([first[v] for v in lab], np.int32)


def _planted(rng, n):
    """Channel 1 of one commit: planted groups (inside ~ U(0.5, 1), across ~ U(0, 0.5), each direction drawn on its own) or
    uniform noise."""
    if rng.random() < 0.3:
        return rng.random((n, n)).astype(np.float32)
    k = int(rng.integers(1, max(2, n // 3) + 1))
    g = rng.integers(0, k, size=n)
    same = g[:, None] == g[None, :]
    return np.where(same, rng.uniform(0.5, 1.0, (n, n)), rng.uniform(0.0, 0.5, (n, n))).astype(np.float32)


def test_oracle_equals_scipy_average_linkage():
    rng = np.random.default_rng(2024)
    compared, rejected, merged, split = 0, 0, 0, 0
    while compared < 80:
        n = int(rng.integers(2, 41))
        P1 = _planted(rng, n)
        thr = float(rng.uniform(0.3, 0.7))
        probs = _probs_of(P1[None])
        w = np.fmax(P1, P1.T).astype(np.float64)
        np.fill_diagonal(w, 1.0)
        Z = linkage(squareform(1.0 - w, checks=False), "average")
        h = np.sort(Z[:, 2])
        # fp32 sums against scipy's fp64: only a comparison whose decisions are 1e-5 apart from each other and from the cut
        # is meaningful; a draw that is not is replaced (and counted)
        if (np.diff(h) <= 1e-5).any() or (np.abs(h - (1.0 - thr)) <= 1e-5).any():
            rejected += 1
            continue
        assert (np.diff(h) > 1e-5).all() and (np.abs(h - (1.0 - thr)) > 1e-5).all()
        ref = _smallest_index_labels(fcluster(Z, t=1.0 - thr, criterion="distance"))
        got, ng = hunk_clusters(probs, None, thr)
        assert np.array_equal(got[0], ref), (n, thr)
        assert ng[0] == len(set(ref.tolist()))
        compared += 1
        merged += ng[0] < n
        split += ng[0] > 1
    assert rejected < 20
    assert merged > 25 and split > 25            # the cuts merge and leave apart: neither side is vacuous


def test_one_confident_pair_does_not_chain_two_groups():
    n = 20
    g = np.repeat([0, 1], 10)
    P1 = np.where(g[:, None] == g[None, :], 0.9, 0.05).astype(np.float32)
    P1[3, 14] = 0.95                                  # one confident false positive between the groups
    probs = _probs_of(P1[None])
    got, ng = hunk_clusters(probs, None, 0.5)
    # the pair is the closest one, so it merges first; its mean with either group, (0.9 + 0.05) / 2, stays below the threshold,
    # so it cannot pull the groups together: one cross pair joined instead of all 100
    want = np.repeat([0, 10], 10)
    want[3] = want[14] = 3
    assert np.array_equal(got[0], want) and ng[0] == 3
    A = (P1 > 1 - P1).astype(np.uint8)                # arg-max relations, p0 = 1 - p1
    np.fill_diagonal(A, 0)
    k, _ = connected_components(csr_matrix(A), directed=True, connection="weak")
    assert k == 1                                     # connected components join them


def test_oracle_threshold_padding_and_nan():
    rng = np.random.default_rng(5)
    n, m = 12, 9
    P1 = _planted(rng, n)
    p1 = _probs_of(P1[None])[0, 1]
    groups, ng = hunk_clusters_one(p1, n, m, 1.0)             # no mean of probabilities in [0, 1] is > 1
    assert np.array_equal(groups, np.arange(n)) and ng == n
    groups, ng = hunk_clusters_one(p1, n, m, -0.5)            # every mean is > -0.5: one group of the real hunks
    assert np.array_equal(groups, np.r_[np.zeros(m), np.arange(m, n)]) and ng == n - m + 1
    junk = P1.copy()
    junk[m:, :] = np.nan
    junk[:, m:] = 7.0
    base = hunk_clusters_one(p1, n, m, 0.5)
    other = hunk_clusters_one(_probs_of(junk[None])[0, 1], n, m, 0.5)
    assert np.array_equal(base[0], other[0]) and base[1] == other[1]
    g, ng = hunk_clusters_one(p1, n, n + 1, 0.5)
    assert (g == -1).all() and ng == -1
    # a pair NaN in both directions keeps its two hunks apart for good; in one direction only the other one counts
    P1 = np.full((4, 4), 0.9, np.float32)
    P1[0, 1] = P1[1, 0] = np.nan
    g, _ = hunk_clusters_one(_probs_of(P1[None])[0, 1], 4, 4, 0.5)
    assert g[0] != g[1]
    P1[1, 0] = 0.9
    g, ng = hunk_clusters_one(_probs_of(P1[None])[0, 1], 4, 4, 0.5)
    assert (g == 0).all() and ng == 1
