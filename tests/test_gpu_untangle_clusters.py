"""GPU tests of the average-linkage hunk clusters: hdgnn_hunk_clusters bit for bit against the NumPy restatement of its
specification (oracle/hunk_clusters.py) in groups and ngroups, with the commit's table in shared memory and in the workspace,
every form of nh, garbage and NaN on the padding pairs, NaN on real pairs, extreme thresholds, many commits per launch,
run-to-run identity, CUDA-graph capture, and graph2graph.untangle(grouping="average") end to end."""
import os

import joblib
import numpy as np
import pytest
import torch

from hdgnn_b200 import _lib
from hdgnn_b200.EvaluationFuncs import partition_metrics_from_counts
from hdgnn_b200.engine import hunk_clusters, pack_label_bits, partition_counts
from hdgnn_b200.synthetic import make_commits
from oracle.hunk_clusters import hunk_clusters as oracle_clusters
from oracle.hunk_clusters import pair_index

pytestmark = pytest.mark.gpu


def planted_probs(rng, B, n, group=8, p_miss=0.15, p_false=0.01):
    """(B, 2, n(n-1)) float32: channel 1 of planted groups of about `group` hunks (inside ~ U(0.55, 0.95), a fraction p_miss of
    the inner pairs missing at ~ U(0, 0.3)), across ~ U(0, 0.35) with a fraction p_false of confident false positives
    ~ U(0.8, 1); both directions drawn on their own; channel 0 = 1 - channel 1."""
    idx = pair_index(n)
    off = idx >= 0
    out = np.empty((B, 2, n * (n - 1)), np.float32)
    for b in range(B):
        g = rng.permutation(n) // group
        same = g[:, None] == g[None, :]
        P = np.where(same, rng.uniform(0.55, 0.95, (n, n)), rng.uniform(0.0, 0.35, (n, n)))
        P = np.where(same & (rng.random((n, n)) < p_miss), rng.uniform(0.0, 0.3, (n, n)), P)
        P = np.where(~same & (rng.random((n, n)) < p_false), rng.uniform(0.8, 1.0, (n, n)), P)
        out[b, 1, idx[off]] = P[off]
    out[:, 0] = 1 - out[:, 1]
    return out


def _run(probs, nh=None, threshold=0.5):
    t = torch.as_tensor(np.ascontiguousarray(probs, dtype=np.float32)).cuda()
    g, ng = hunk_clusters(t, None if nh is None else torch.as_tensor(np.asarray(nh, np.int32)).cuda(), threshold)
    return g.cpu().numpy(), ng.cpu().numpy()


def _check(probs, nh=None, threshold=0.5):
    got = _run(probs, nh, threshold)
    ref = oracle_clusters(probs, nh, threshold)
    for b in range(probs.shape[0]):
        assert np.array_equal(got[0][b], ref[0][b]), (b, None if nh is None else nh[b])
    assert np.array_equal(got[1], ref[1])
    return got


def _padding_junk(rng, probs, nh):
    """probs with every pair that touches a hunk >= nh[b] overwritten by random values and NaNs, in both channels."""
    probs = probs.copy()
    B, _, ncr = probs.shape
    n = (1 + int(round((1 + 4 * ncr) ** 0.5))) // 2
    idx = pair_index(n)
    for b in range(B):
        m = int(nh[b])
        touch = (idx >= 0) & ((np.arange(n)[:, None] >= m) | (np.arange(n)[None, :] >= m))
        p = idx[touch]
        junk = rng.uniform(-2, 3, size=(2, p.size)).astype(np.float32)
        junk[rng.random((2, p.size)) < 0.3] = np.nan
        probs[b][:, p] = junk
    return probs


@pytest.mark.parametrize("n", [2, 3, 31, 32, 33, 74, 150, 256, 300, 512])
def test_hunk_clusters_equal_the_oracle(n):
    rng = np.random.default_rng(900 + n)
    in_smem = _lib.lib.hdgnn_hunk_clusters_work(8, n) == 0
    assert in_smem == (n <= 169)                                  # both sides of the shared-memory / workspace split
    B = 8 if n <= 256 else 5
    probs = planted_probs(rng, B, n)
    g, ng = _check(probs)                                         # nh = None: every hunk is real
    if n >= 74:
        assert (ng > 1).all() and (ng < n).all()                  # the planted groups are found, not all or nothing
    # nh random, 0, 1, n and out of range (rows of -1); the padding pairs hold random values and NaNs
    nh = np.concatenate([[0, 1, n, -1, n + 1], rng.integers(0, n + 1, size=B)]).astype(np.int32)[:max(B, 5)]
    probs = planted_probs(rng, len(nh), n)
    gn, ngn = _check(probs, nh)
    bad = (nh < 0) | (nh > n)
    assert (gn[bad] == -1).all() and (ngn[bad] == -1).all()
    assert np.array_equal(gn[nh == 0][:, :], np.tile(np.arange(n, dtype=np.int32), ((nh == 0).sum(), 1)))
    junk = _padding_junk(rng, probs, np.clip(nh, 0, n))
    gj, ngj = _run(junk, nh)
    assert np.array_equal(gj, gn) and np.array_equal(ngj, ngn)   # pairs of padding hunks are never read
    gr, ngr = _run(probs, nh)
    assert np.array_equal(gr, gn) and np.array_equal(ngr, ngn)   # run to run


@pytest.mark.parametrize("n", [33, 256])
def test_thresholds_and_nan_pairs(n):
    rng = np.random.default_rng(40 + n)
    B = 4
    probs = planted_probs(rng, B, n)
    nh = np.array([n, n - 3, 5, 2], np.int32)
    g, ng = _run(probs, nh, 1.0)                                  # no mean of probabilities in [0, 1] is > 1: singletons
    assert np.array_equal(g, np.tile(np.arange(n, dtype=np.int32), (B, 1))) and (ng == n).all()
    g, ng = _run(probs, nh, -0.25)                                # every mean is > -0.25: one group of the real hunks
    for b in range(B):
        assert (g[b, :nh[b]] == 0).all() and np.array_equal(g[b, nh[b]:], np.arange(nh[b], n)) and ng[b] == n - nh[b] + 1
    _check(probs, nh, 1.0)
    _check(probs, nh, -0.25)
    # NaN on real pairs: in one direction (the other one counts) and in both (the two hunks never share a group)
    idx = pair_index(n)
    for b in range(B):
        m = int(nh[b])
        for _ in range(max(1, m // 4)):
            s, t = rng.choice(m, 2, replace=False)
            probs[b, 1, idx[s, t]] = np.nan
            if rng.random() < 0.5:
                probs[b, 1, idx[t, s]] = np.nan
    for thr in (0.5, 0.3, -0.25):
        _check(probs, nh, thr)


def test_hunk_clusters_of_many_commits():
    """1001 commits at 74 (one CTA each, table in shared memory) and 400 at 512 (persistent CTAs walking the commits, one
    workspace slice each)."""
    for n, B, step in ((74, 1001, 37), (512, 400, 97)):
        rng = np.random.default_rng(n + B)
        probs = planted_probs(rng, B, n)
        nh = rng.integers(n // 2, n + 1, size=B).astype(np.int32)
        g, ng = _run(probs, nh)
        pick = list(range(0, B, step)) + [B - 1]
        ref = oracle_clusters(probs[pick], nh[pick], 0.5)
        assert np.array_equal(g[pick], ref[0]) and np.array_equal(ng[pick], ref[1]), n


def test_hunk_clusters_in_a_cuda_graph():
    rng = np.random.default_rng(3)
    for n, B in ((74, 300), (300, 20)):
        probs = torch.as_tensor(planted_probs(rng, B, n)).cuda()
        nh = torch.as_tensor(rng.integers(0, n + 1, size=B).astype(np.int32)).cuda()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            hunk_clusters(probs, nh, 0.5)                                  # warm-up outside the capture
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            groups, ngroups = hunk_clusters(probs, nh, 0.5)
        probs.copy_(torch.as_tensor(planted_probs(rng, B, n)))
        g.replay()
        torch.cuda.synchronize()
        ref = oracle_clusters(probs.cpu().numpy(), nh.cpu().numpy(), 0.5)
        assert np.array_equal(groups.cpu().numpy(), ref[0]) and np.array_equal(ngroups.cpu().numpy(), ref[1])


def test_hunk_clusters_rejects_bad_tensors():
    p = torch.zeros(2, 2, 74 * 73, device="cuda")
    with pytest.raises(ValueError):
        hunk_clusters(p[:, :, :-1])                                       # not n(n-1) pairs
    with pytest.raises(ValueError):
        hunk_clusters(p.double())
    with pytest.raises(ValueError):
        hunk_clusters(p, torch.zeros(3, dtype=torch.int32, device="cuda"))
    with pytest.raises(RuntimeError):
        hunk_clusters(p.cpu())
    with pytest.raises(_lib.HdgnnError):
        hunk_clusters(p, None, float("nan"))


# ---- graph2graph.untangle(grouping="average") end to end --------------------------------------------------------------
def _argmax_bits(probs: np.ndarray, Nc: int) -> np.ndarray:
    B = probs.shape[0]
    grid = np.zeros((B, Nc, Nc), dtype=np.uint8)
    grid[:, ~np.eye(Nc, dtype=bool)] = probs[:, 1] > probs[:, 0]
    return pack_label_bits(grid)


def test_untangle_average_linkage_after_train(tmp_path):
    from hdgnn_b200.model import graph2graph
    from hdgnn_b200.utils2 import write_dataset, read_compact, split_half
    Ne, Nc, N, MB = 12, 8, 16, 4
    cb = make_commits(N, Ne, Nc, seed=8, p_edge=0.2, p_short=0.4, p_noise=0.2)
    keep = [None] * N
    for b in range(N):                      # commits with fewer than Nc hunks: the rest of their grid is padding
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
    with pytest.raises(ValueError):
        model.untangle(None, root=root, log=lambda s: None, grouping="single")
    _, probs = model.test(None, root=root, log=lambda s: None)
    n = test.B
    nh = test.nh[:n].astype(np.int32)
    pt = torch.as_tensor(np.ascontiguousarray(probs)).cuda()
    thr = float(np.median(probs[:, 1]))                # a threshold the trained model's probabilities straddle
    for threshold in (0.5, thr):
        logs = []
        out = model.untangle(None, root=root, log=logs.append, grouping="average", threshold=threshold)
        ref, _ = hunk_clusters(pt, torch.as_tensor(nh).cuda(), threshold)
        ref = ref.cpu().numpy()
        assert np.array_equal(out["groups"], ref)
        d = tmp_path / "outputSelf" / "toy" / "model_2" / "2"
        assert np.array_equal(np.load(d / f"C_group_t{Ne}.npy"), ref)
        assert np.array_equal(out["pred_bits"].view(np.uint32), _argmax_bits(probs, Nc))
        assert np.array_equal(out["label_groups"], np.load(d / f"C_group_y{Ne}.npy"))   # labelled groups as before
        lab = torch.as_tensor(out["label_groups"]).cuda()
        want = partition_counts(torch.as_tensor(ref).cuda(), lab, torch.as_tensor(nh).cuda()).cpu().numpy()
        assert np.array_equal(out["partition_counts"], want)
        assert out["partition"] == partition_metrics_from_counts(want)
        assert out["exact_partitions"] == int((ref == out["label_groups"]).all(1).sum())
        k = len(out["partition"])
        assert logs[-3 - k] == f"grouping: average linkage, threshold {threshold}"
        assert logs[-2 - k:-2] == [f"partition_{key}: {v}" for key, v in out["partition"].items()]
        assert logs[-2].startswith("exact_partitions: ") and logs[-1].startswith("test time:")
    model.engine.close()
