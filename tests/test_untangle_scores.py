"""CPU checks of the untangling scores: EvaluationFuncs.partition_metrics_from_counts agrees with sklearn.metrics, and the
loader reads, caches and reloads the number of real hunks per commit (CommitBatch.nh)."""
import os

import joblib
import numpy as np
import pytest
from sklearn.metrics import adjusted_rand_score, pair_confusion_matrix, rand_score
from sklearn.metrics.cluster import contingency_matrix

from hdgnn_b200.EvaluationFuncs import partition_metrics_from_counts


# ---- metrics against sklearn --------------------------------------------------------------------------------------
def host_counts(pred, truth):
    """The eight counters of hdgnn_partition_counts for one commit's real hunks, from sklearn's contingency table."""
    m = len(pred)
    if m == 0:
        return np.zeros(8, np.int64)
    Cm = contingency_matrix(truth, pred)             # rows: truth groups, columns: pred groups
    pairs = lambda x: int((x * (x - 1) // 2).sum())
    return np.array([m, pairs(Cm), pairs(Cm.sum(0)), pairs(Cm.sum(1)), Cm.shape[1], Cm.shape[0],
                     Cm.max(0).sum(), Cm.max(1).sum()], np.int64)


def _partition(rng, m, k):
    """m hunks in at most k groups under arbitrary (non-canonical) label values."""
    names = rng.permutation(10 * max(k, 1))[:k] + 7
    return names[rng.integers(0, k, size=m)]


def _cases(rng):
    """(pred, truth) pairs: all singletons, one group, m = 0 / 1 / 2, identical partitions, random ones of every size."""
    out = [(np.arange(9), np.arange(9)), (np.zeros(9, int), np.zeros(9, int)), (np.arange(9), np.zeros(9, int)),
           (np.zeros(9, int), np.arange(9)), (np.zeros(0, int), np.zeros(0, int)), (np.array([3]), np.array([5])),
           (np.array([0, 0]), np.array([1, 1])), (np.array([0, 1]), np.array([4, 4])), (np.array([2, 3]), np.array([0, 1]))]
    same = _partition(rng, 40, 6)
    out.append((same, rng.permutation(100)[same]))    # the same partition under other names
    for m in (3, 5, 17, 74, 200):
        for k in (1, 2, max(2, m // 4), m):
            out.append((_partition(rng, m, k), _partition(rng, m, max(1, k // 2 + 1))))
    return out


def test_host_counters_agree_with_the_pair_confusion_matrix():
    for p, t in _cases(np.random.default_rng(1)):
        c = host_counts(p, t)
        if len(p) < 2:
            continue
        (tn, fp), (fn, tp) = pair_confusion_matrix(t, p) // 2          # ordered pairs -> unordered
        assert (c[1], c[2], c[3]) == (tp, tp + fp, tp + fn)
        assert tn + fp + fn + tp == len(p) * (len(p) - 1) // 2


def test_partition_metrics_agree_with_sklearn():
    cases = _cases(np.random.default_rng(2))
    counts = np.stack([host_counts(p, t) for p, t in cases])
    got = partition_metrics_from_counts(counts)
    big = [(p, t) for p, t in cases if len(p) >= 2]
    assert got["commits"] == len(cases)
    assert got["exact"] == sum(adjusted_rand_score(t, p) == 1.0 for p, t in cases if len(p) >= 2) + sum(len(p) < 2 for p, _ in cases)
    assert got["rand"] == pytest.approx(np.mean([rand_score(t, p) for p, t in big]), rel=1e-12)
    assert got["ari"] == pytest.approx(np.mean([adjusted_rand_score(t, p) for p, t in big]), rel=1e-12)
    pcm = sum(pair_confusion_matrix(t, p) for p, t in big) // 2
    tp, fp, fn = pcm[1, 1], pcm[0, 1], pcm[1, 0]
    assert got["pair_precision"] == pytest.approx(tp / (tp + fp), rel=1e-12)
    assert got["pair_recall"] == pytest.approx(tp / (tp + fn), rel=1e-12)
    assert got["pair_f1"] == pytest.approx(2 * tp / (2 * tp + fp + fn), rel=1e-12)
    hunks = sum(len(p) for p, _ in cases)
    assert got["purity"] == pytest.approx(sum(contingency_matrix(t, p).max(0).sum() for p, t in cases if len(p)) / hunks)
    assert got["inverse_purity"] == pytest.approx(sum(contingency_matrix(t, p).max(1).sum() for p, t in cases if len(p)) / hunks)
    assert got["groups_pred_mean"] == pytest.approx(np.mean([len(np.unique(p)) for p, _ in cases]))
    assert got["groups_truth_mean"] == pytest.approx(np.mean([len(np.unique(t)) for _, t in cases]))
    # one commit at a time: sklearn's own value, its 1.0 for partitions without a disagreeing pair included
    for p, t in big:
        one = partition_metrics_from_counts(host_counts(p, t)[None])
        assert one["rand"] == rand_score(t, p) and one["ari"] == adjusted_rand_score(t, p), (p, t)
        assert one["exact"] == int(adjusted_rand_score(t, p) == 1.0)


def test_partition_metrics_edge_cases():
    empty = partition_metrics_from_counts(np.zeros((0, 8), np.int64))
    assert empty["commits"] == 0 and empty["exact"] == 0 and empty["pair_f1"] == 0.0 and empty["purity"] == 0.0
    assert np.isnan(empty["rand"]) and np.isnan(empty["ari"])
    small = partition_metrics_from_counts(np.stack([host_counts(np.zeros(0, int), np.zeros(0, int)),
                                                    host_counts(np.array([1]), np.array([2]))]))
    assert small["exact"] == 2 and np.isnan(small["rand"]) and small["pair_precision"] == 0.0 and small["purity"] == 1.0
    singles = partition_metrics_from_counts(host_counts(np.arange(5), np.arange(5))[None])
    assert singles["pair_precision"] == 0.0 and singles["pair_recall"] == 0.0 and singles["ari"] == 1.0 and singles["rand"] == 1.0
    c = np.stack([host_counts(np.arange(5), np.zeros(5, int)), np.full(8, -1)])
    with pytest.raises(ValueError):
        partition_metrics_from_counts(c)


# ---- the loader's hunk counts --------------------------------------------------------------------------------------
def shorten_maps(repo, step, root, keep):
    """Rewrite the HunkIDmap pickle of a write_dataset tree so that commit b's map holds hunk numbers 0 .. keep[b]-1 only
    (keep[b] None: the map is left as written).  No entity line of commit b may name a hunk >= keep[b]."""
    path = os.path.join(root, "dataset", repo, "HunkIDdict", f"HunkIDmap_{step}.pkl")
    maps = joblib.load(path)
    for b, k in enumerate(keep):
        if k is not None:
            maps[b] = {key: v for key, v in maps[b].items() if v < k}
    joblib.dump(maps, path)


def test_loader_reads_caches_and_reloads_the_hunk_counts(tmp_path):
    from hdgnn_b200.synthetic import make_commits
    from hdgnn_b200.utils2 import read_compact, write_dataset, _cache_path
    Ne, Nc, N = 10, 6, 6
    cb = make_commits(N, Ne, Nc, seed=4)
    keep = [None, 0, 1, 3, Nc, Nc + 2]
    for b, k in enumerate(keep):
        if k is not None:
            cb.hmap[b][cb.hmap[b] >= k] = -1
    root = str(tmp_path)
    write_dataset(cb, "toy", 3, root=root)
    shorten_maps("toy", 3, root, keep)
    want = np.array([Nc, 0, 1, 3, Nc, Nc], np.int32)
    got = read_compact("toy", 3, Ne, Nc, root=root)
    assert got.nh.dtype == np.int32 and np.array_equal(got.nh, want)
    assert np.array_equal(got.slice(2, 5).nh, want[2:5])
    cached = read_compact("toy", 3, Ne, Nc, root=root)                 # the cache written by the first call
    assert np.array_equal(cached.nh, want) and np.array_equal(cached.Y, got.Y)
    cp = _cache_path(root, "toy", 3, Ne, Nc)
    np.savez_compressed(cp, adj=got.adj, x=got.x, hmap=got.hmap, L=got.L, Y=got.Y)     # a cache from before the hunk counts
    old = read_compact("toy", 3, Ne, Nc, root=root)
    assert old.nh is None and np.array_equal(old.hmap, got.hmap) and old.slice(0, 2).nh is None
