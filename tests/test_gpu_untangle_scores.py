"""GPU tests of the untangling scores: hdgnn_partition_counts against a host computation from sklearn's contingency table (any
labels, partitions of hunk_groups, every form of nh, garbage on the padding hunks), rows of -1 for commits it cannot score,
batches of several commits per CTA, determinism, CUDA-graph capture, and graph2graph.untangle end to end on a data set whose
hunk maps leave some commits with fewer than Nc hunks.  Every counter comparison is integer and exact."""
import os

import joblib
import numpy as np
import pytest
import torch
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components
from sklearn.metrics.cluster import contingency_matrix

from hdgnn_b200.EvaluationFuncs import partition_metrics_from_counts
from hdgnn_b200.engine import hunk_groups, pack_label_bits, partition_counts
from hdgnn_b200.synthetic import make_commits

pytestmark = pytest.mark.gpu


def host_counts(pred, truth, nh=None):
    """(B, n) labels -> (B, 8) counters of hdgnn_partition_counts over the first nh[b] hunks (all n if nh is None)."""
    B, n = pred.shape
    out = np.zeros((B, 8), np.int64)
    for b in range(B):
        m = n if nh is None else int(nh[b])
        if m < 0 or m > n or ((pred[b, :m] < 0) | (pred[b, :m] >= n) | (truth[b, :m] < 0) | (truth[b, :m] >= n)).any():
            out[b] = -1
            continue
        if m == 0:
            continue
        Cm = contingency_matrix(truth[b, :m], pred[b, :m])
        pairs = lambda x: int((x * (x - 1) // 2).sum())
        out[b] = [m, pairs(Cm), pairs(Cm.sum(0)), pairs(Cm.sum(1)), Cm.shape[1], Cm.shape[0], Cm.max(0).sum(), Cm.max(1).sum()]
    return out


def _labels(rng, B, n):
    """Arbitrary label values in [0, n): per commit k groups under random names, k from 1 to n."""
    out = np.empty((B, n), np.int32)
    for b in range(B):
        k = int(rng.choice([1, 2, max(1, n // 8), max(1, n // 2), n]))
        names = rng.permutation(n)[:k]
        out[b] = names[rng.integers(0, k, size=n)]
    return out


def _groups_of_random_graphs(rng, B, n, p):
    A = (rng.random((B, n, n)) < p).astype(np.uint8)
    g, _ = hunk_groups(torch.as_tensor(pack_label_bits(A).view(np.int32)).cuda())
    return g.cpu().numpy()


def _garbage_padding(rng, x, nh):
    """x with the hunks >= nh[b] overwritten by anything, out-of-range values included."""
    x = x.copy()
    B, n = x.shape
    junk = rng.choice(np.array([-1, -7, n, n + 5, 2 ** 31 - 1, -2 ** 31, 0, n - 1], np.int64), size=(B, n)).astype(np.int32)
    pad = np.arange(n)[None, :] >= nh[:, None]
    x[pad] = junk[pad]
    return x


def _run(pred, truth, nh=None):
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).cuda()
    return partition_counts(t(pred), t(truth), None if nh is None else t(nh)).cpu().numpy()


@pytest.mark.parametrize("n", [2, 31, 32, 33, 74, 150, 256, 300, 512])
def test_partition_counts_equal_the_host(n):
    rng = np.random.default_rng(500 + n)
    B = 24
    rand_p, rand_t = _labels(rng, B, n), _labels(rng, B, n)
    hg_p = _groups_of_random_graphs(rng, B, n, 1.0 / n)
    hg_t = _groups_of_random_graphs(rng, B, n, 1.5 / n)
    hg_t[: B // 4] = hg_p[: B // 4]                                              # identical partitions
    fixed = np.array([0, 1, 2, n, min(3, n), n - 1], np.int32)
    nh = np.concatenate([fixed, rng.integers(0, n + 1, size=B - len(fixed))]).astype(np.int32)
    for pred, truth in ((rand_p, rand_t), (hg_p, hg_t), (rand_p, hg_t)):
        got = _run(pred, truth)                                                  # nh = None: every hunk is real
        assert np.array_equal(got, host_counts(pred, truth)), n
        assert (got[:, 0] == n).all()
        gp, gt = _garbage_padding(rng, pred, nh), _garbage_padding(rng, truth, nh)
        got = _run(gp, gt, nh)
        assert np.array_equal(got, host_counts(pred, truth, nh)), n
        assert np.array_equal(got, _run(gp, gt, nh))                            # deterministic
    full = _run(hg_p, hg_p, np.full(B, n, np.int32))
    assert (full[:, 1] == full[:, 2]).all() and (full[:, 2] == full[:, 3]).all() and (full[:, 6] == n).all()


def test_invalid_commits_get_a_row_of_minus_one_and_only_they():
    rng = np.random.default_rng(7)
    B, n = 8, 74
    pred, truth = _labels(rng, B, n), _labels(rng, B, n)
    nh = np.full(B, 40, np.int32)
    pred[1, 39] = n                           # out of range on the last real hunk
    truth[2, 0] = -1
    nh[3], nh[4] = -1, n + 1                  # hunk counts outside [0, n]
    pred[5, 40] = n + 9                       # out of range on a padding hunk: no effect
    got = _run(pred, truth, nh)
    assert (got[1:5] == -1).all()
    keep = [0, 5, 6, 7]
    assert np.array_equal(got[keep], host_counts(pred[keep], truth[keep], nh[keep]))
    assert (got[keep] >= 0).all()


def test_partition_counts_of_many_commits():
    """Batches that put several commits into one CTA (1001 at 74: the last CTA has idle warps; 400 at 512: two 76 KB commits)."""
    for n, B in ((74, 1001), (512, 400), (74, 4096)):
        rng = np.random.default_rng(n + B)
        pred, truth = _labels(rng, B, n), _labels(rng, B, n)
        nh = rng.integers(0, n + 1, size=B).astype(np.int32)
        got = _run(pred, truth, nh)
        for b in range(0, B, 23):
            assert np.array_equal(got[b], host_counts(pred[b:b + 1], truth[b:b + 1], nh[b:b + 1])[0]), (n, B, b)


def test_partition_counts_in_a_cuda_graph():
    rng = np.random.default_rng(3)
    for n, B in ((74, 300), (512, 50)):
        pred = torch.as_tensor(_labels(rng, B, n)).cuda()
        truth = torch.as_tensor(_labels(rng, B, n)).cuda()
        nh = torch.as_tensor(rng.integers(0, n + 1, size=B).astype(np.int32)).cuda()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            partition_counts(pred, truth, nh)                                   # warm-up outside the capture
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = partition_counts(pred, truth, nh)
        pred.copy_(torch.as_tensor(_labels(rng, B, n)))
        g.replay()
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), host_counts(pred.cpu().numpy(), truth.cpu().numpy(), nh.cpu().numpy()))


# ---- graph2graph.untangle end to end ---------------------------------------------------------------------------
def _scipy_groups(A: np.ndarray):
    n = A.shape[0]
    A = A.copy()
    np.fill_diagonal(A, 0)
    k, lab = connected_components(csr_matrix(A), directed=True, connection="weak")
    first = np.full(k, n, dtype=np.int64)
    np.minimum.at(first, lab, np.arange(n))
    return first[lab].astype(np.int32)


def test_untangle_scores_the_real_hunks(tmp_path):
    from hdgnn_b200.model import graph2graph
    from hdgnn_b200.utils2 import write_dataset, read_compact, split_half
    Ne, Nc, N, MB = 12, 8, 16, 4
    cb = make_commits(N, Ne, Nc, seed=8, p_edge=0.2, p_short=0.4, p_noise=0.2)
    keep = [None] * N
    for b in range(N):                      # commits of both halves with fewer than Nc hunks: the rest of their grid is padding
        k = [3, 5, None, 2][b % 4]
        if k is not None:
            keep[b] = k
            cb.hmap[b][cb.hmap[b] >= k] = -1
            cb.Y[b, k:, :] = 0
            cb.Y[b, :, k:] = 0
    root = str(tmp_path)
    write_dataset(cb, "toy", 2, root=root)
    path = os.path.join(root, "dataset", "toy", "HunkIDdict", "HunkIDmap_2.pkl")
    maps = joblib.load(path)
    maps = [m if k is None else {key: v for key, v in m.items() if v < k} for m, k in zip(maps, keep)]
    joblib.dump(maps, path)
    _, test = split_half(read_compact("toy", 2, Ne, Nc, root=root))
    assert test.nh is not None and (test.nh < Nc).any()
    model = graph2graph(None, Ne=Ne, Nc=Nc, Mini_batch=MB, epoch=3, Step=2, Repo="toy", variant=2, seed=11,
                        checkpoint_dir=str(tmp_path / "ck"))
    model.train(None, root=root, log=lambda s: None)
    logs = []
    out = model.untangle(None, root=root, log=logs.append)
    n = test.B
    # unchanged outputs: the files, the groups over all Nc hunks, exact_partitions and the last two log lines
    d = tmp_path / "outputSelf" / "toy" / "model_2" / "2"
    gt, gy = np.load(d / f"C_group_t{Ne}.npy"), np.load(d / f"C_group_y{Ne}.npy")
    assert gt.shape == (n, Nc) and gt.dtype == np.int32 and gy.dtype == np.int32
    assert np.array_equal(gy, np.stack([_scipy_groups(test.Y[k]) for k in range(n)]))
    ref, _ = hunk_groups(torch.as_tensor(out["pred_bits"]).cuda())
    assert np.array_equal(gt, ref.cpu().numpy())
    assert np.array_equal(out["groups"], gt) and np.array_equal(out["label_groups"], gy)
    assert out["exact_partitions"] == int((gt == gy).all(1).sum())
    assert logs[-2] == f"exact_partitions: {out['exact_partitions']} / {n}" and logs[-1].startswith("test time:")
    # the scores: over the real hunks of each commit, from the loader's hunk counts
    want = host_counts(gt, gy, test.nh[:n])
    assert np.array_equal(out["partition_counts"], want)
    assert out["partition"] == partition_metrics_from_counts(want)
    unmasked = host_counts(gt, gy)
    assert (unmasked != want).any(axis=1).any()
    assert partition_metrics_from_counts(unmasked) != out["partition"]
    lines = logs[-2 - len(out["partition"]):-2]
    assert lines == [f"partition_{k}: {v}" for k, v in out["partition"].items()]
    model.engine.close()
