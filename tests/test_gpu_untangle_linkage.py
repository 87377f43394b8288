"""GPU tests of the average-linkage dendrogram: hdgnn_hunk_linkage bit for bit against the oracle's merge record
(tests/linkage_oracle.py) on both sides of the shared-memory / workspace split, with every form of nh, garbage and NaN on the
padding pairs and NaN on real pairs, and beyond the 296 workspace slices; hdgnn_linkage_cut bit for bit against
hdgnn_hunk_clusters at every recorded height, one ulp either side, +-inf, 0 and 1, and against the oracle at a group count;
corrupted records; CUDA-graph capture; graph2graph.untangle(sweep=...) end to end."""
import numpy as np
import pytest
import torch

from hdgnn_b200 import _lib
from hdgnn_b200.EvaluationFuncs import partition_metrics_from_counts
from hdgnn_b200.engine import hunk_clusters, hunk_linkage, linkage_cut, partition_counts
from linkage_oracle import hunk_linkage as oracle_linkage
from linkage_oracle import linkage_cut as oracle_cut
from oracle.hunk_clusters import pair_index
from test_gpu_untangle_clusters import _padding_junk, planted_probs

pytestmark = pytest.mark.gpu


def _cuda(x):
    return None if x is None else torch.as_tensor(np.ascontiguousarray(x)).cuda()


def _run(probs, nh=None):
    return tuple(x.cpu().numpy() for x in hunk_linkage(_cuda(probs), _cuda(None if nh is None else np.asarray(nh, np.int32))))


def _same_record(got, ref):
    """merges and nmerges equal; heights equal bit for bit where recorded, NaN where not."""
    (gm, gh, gn), (rm, rh, rn) = got, ref
    assert np.array_equal(gn, rn)
    assert np.array_equal(gm, rm)
    assert np.array_equal(np.isnan(gh), np.isnan(rh))
    ok = ~np.isnan(rh)
    assert np.array_equal(gh[ok].view(np.int32), rh[ok].view(np.int32))


def _nan_pairs(rng, probs, nh):
    probs = probs.copy()
    n = (1 + int(round((1 + 4 * probs.shape[2]) ** 0.5))) // 2
    idx = pair_index(n)
    for b in range(probs.shape[0]):
        m = int(nh[b]) if 0 <= nh[b] <= n else 0
        for i in range(m // 8 if m >= 3 else 0):
            s, t = rng.choice(m, 2, replace=False)
            probs[b, 1, idx[s, t]] = np.nan
            if i == 0 or rng.random() < 0.5:                        # NaN both ways: s and t never join
                probs[b, 1, idx[t, s]] = np.nan
    return probs


@pytest.mark.parametrize("n", [2, 3, 31, 32, 33, 74, 128, 169, 170, 256, 512])
def test_hunk_linkage_equals_the_oracle(n):
    rng = np.random.default_rng(1200 + n)
    assert (_lib.lib.hdgnn_hunk_clusters_work(8, n) == 0) == (n <= 169)
    B = 6 if n <= 170 else 3
    probs = planted_probs(rng, B, n)
    _same_record(_run(probs), oracle_linkage(probs))
    # every form of nh: 0, 1, m < n, n, out of range; the padding pairs hold random values and NaNs; NaN on real pairs
    nh = np.array([0, 1, max(n - 3, 0), n, -1, n + 1], np.int32)
    probs = _nan_pairs(rng, planted_probs(rng, len(nh), n), nh)
    ref = oracle_linkage(probs, nh)
    got = _run(_padding_junk(rng, probs, np.clip(nh, 0, n)), nh)
    _same_record(got, ref)
    bad = (nh < 0) | (nh > n)
    assert (got[2][bad] == -1).all() and (got[0][bad] == -1).all() and np.isnan(got[1][bad]).all()
    if n >= 33:
        assert (got[2][~bad] < np.maximum(nh[~bad] - 1, 0)).any()    # NaN pairs stop a sequence early
    _same_record(_run(probs, nh), got)                               # run to run


def _thresholds(heights, rng, k=24):
    h = np.unique(heights[~np.isnan(heights)].astype(np.float32))
    h = rng.choice(h, min(k, h.size), replace=False) if h.size else h
    extra = np.float32([-np.inf, np.inf, 0.0, 1.0])
    return np.unique(np.r_[h, np.nextafter(h, np.float32(np.inf)), np.nextafter(h, np.float32(-np.inf)), extra])


@pytest.mark.parametrize("n", [33, 74, 256])
def test_linkage_cut_equals_hunk_clusters(n):
    rng = np.random.default_rng(60 + n)
    B = 8
    nh = np.array([n, n, n - 5, 2, 1, 0, n, n // 2], np.int32)
    probs = _nan_pairs(rng, planted_probs(rng, B, n), nh)
    probs[:2, 1] = np.round(probs[:2, 1] * 4) / 4                   # equal means: the tie rule decides
    p, h = _cuda(probs), _cuda(nh)
    rec = hunk_linkage(p, h)
    ts = _thresholds(rec[1].cpu().numpy(), rng)
    for lo in range(0, len(ts), 64):
        chunk = [float(t) for t in ts[lo:lo + 64]]
        g, ng = linkage_cut(*rec, h, thresholds=chunk)
        for k, t in enumerate(chunk):
            rg, rn = hunk_clusters(p, h, t)
            assert torch.equal(g[k], rg) and torch.equal(ng[k], rn), t
    # the group-count cut against the oracle, targets from below 1 to above m
    target = np.array([3, 1, 0, -4, 9, 2, n + 7, 5], np.int32)
    g, ng = linkage_cut(*rec, h, target=_cuda(target))
    rm, rh, rn = (x.cpu().numpy() for x in rec)
    want = oracle_cut(rm, rh, rn, nh, target=target)
    assert np.array_equal(g.cpu().numpy(), want[0]) and np.array_equal(ng.cpu().numpy(), want[1])


def test_linkage_of_many_commits():
    """600 commits: more than the 296 persistent CTAs of the workspace form, which walk the commits."""
    for n in (74, 200):
        rng = np.random.default_rng(n)
        probs = planted_probs(rng, 600, n)
        nh = rng.integers(n // 2, n + 1, size=600).astype(np.int32)
        got = _run(probs, nh)
        pick = [0, 1, 295, 296, 297, 443, 591, 599]
        _same_record(tuple(x[pick] for x in got), oracle_linkage(probs[pick], nh[pick]))
        g, ng = linkage_cut(*(_cuda(x) for x in got), _cuda(nh), thresholds=[0.5])
        rg, rn = hunk_clusters(_cuda(probs), _cuda(nh), 0.5)
        assert torch.equal(g[0], rg) and torch.equal(ng[0], rn)


def test_corrupted_records_give_minus_one_rows():
    rng = np.random.default_rng(9)
    n, B = 40, 7
    probs = planted_probs(rng, B, n)
    m, h, c = (x.cpu().numpy() for x in hunk_linkage(_cuda(probs)))
    assert (c == n - 1).all()
    m[1, 4] = m[1, 4, ::-1]                       # a >= c
    m[2, 9, 1] = m[2, 3, 1]                       # a repeated c
    m[3, 20, 0] = m[3, 2, 1]                      # an a absorbed at an earlier row
    c[4] = n                                      # more merges than m - 1
    m[5, 7, 1] = n + 100                          # c outside the commit
    c[6] = -3
    g, ng = linkage_cut(_cuda(m), _cuda(h), _cuda(c), thresholds=[0.5, -np.inf])
    torch.cuda.synchronize()
    g, ng = g.cpu().numpy(), ng.cpu().numpy()
    assert (g[:, 1:] == -1).all() and (ng[:, 1:] == -1).all()
    assert (g[:, 0] >= 0).all() and (ng[:, 0] > 0).all()
    want = oracle_cut(m, h, c, thresholds=[0.5, -np.inf])
    assert np.array_equal(g, want[0]) and np.array_equal(ng, want[1])
    gt, _ = linkage_cut(_cuda(m), _cuda(h), _cuda(c), target=_cuda(np.full(B, 3, np.int32)))
    assert (gt[0, 1:] == -1).all().item()


def test_linkage_and_cut_in_a_cuda_graph():
    rng = np.random.default_rng(5)
    for n, B in ((74, 300), (300, 20)):
        probs = _cuda(planted_probs(rng, B, n))
        nh = _cuda(rng.integers(0, n + 1, size=B).astype(np.int32))
        ts = [0.9, 0.5, 0.25]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            linkage_cut(*hunk_linkage(probs, nh), nh, thresholds=ts)           # warm-up outside the capture
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            rec = hunk_linkage(probs, nh)
            groups, ngroups = linkage_cut(*rec, nh, thresholds=ts)
        probs.copy_(_cuda(planted_probs(rng, B, n)))
        graph.replay()
        torch.cuda.synchronize()
        first = [x.clone() for x in (*rec, groups, ngroups)]
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(first, (*rec, groups, ngroups)))
        for k, t in enumerate(ts):
            rg, rn = hunk_clusters(probs, nh, t)
            assert torch.equal(groups[k], rg) and torch.equal(ngroups[k], rn)


# ---- graph2graph.untangle(sweep=...) end to end ----------------------------------------------------------------------------
def test_untangle_sweep_after_train(tmp_path):
    import joblib
    import os
    from hdgnn_b200.model import graph2graph
    from hdgnn_b200.synthetic import make_commits
    from hdgnn_b200.utils2 import read_compact, split_half, write_dataset
    Ne, Nc, N, MB = 12, 8, 16, 4                  # the dataset of test_untangle_average_linkage_after_train
    cb = make_commits(N, Ne, Nc, seed=8, p_edge=0.2, p_short=0.4, p_noise=0.2)
    keep = [None] * N
    for b in range(N):
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
    joblib.dump([m if k is None else {key: v for key, v in m.items() if v < k} for m, k in zip(maps, keep)], path)
    _, test = split_half(read_compact("toy", 2, Ne, Nc, root=root))
    model = graph2graph(None, Ne=Ne, Nc=Nc, Mini_batch=MB, epoch=3, Step=2, Repo="toy", variant=2, seed=11,
                        checkpoint_dir=str(tmp_path / "ck"))
    model.train(None, root=root, log=lambda s: None)
    with pytest.raises(ValueError):
        model.untangle(None, root=root, log=lambda s: None, sweep=[0.5])                 # components: no dendrogram
    _, probs = model.test(None, root=root, log=lambda s: None)
    n = test.B
    nh = _cuda(test.nh[:n].astype(np.int32))
    pt = _cuda(probs)
    d = tmp_path / "outputSelf" / "toy" / "model_2" / "2"
    thr = float(np.median(probs[:, 1]))
    sweep = [0.9, thr, 0.5, 0.1, -1.0]
    plain_logs, logs = [], []
    plain = model.untangle(None, root=root, log=plain_logs.append, grouping="average", threshold=thr)
    plain_files = {f: np.load(d / f"{f}{Ne}.npy") for f in ("C_group_t", "C_group_y")}
    out = model.untangle(None, root=root, log=logs.append, grouping="average", threshold=thr, sweep=sweep)
    for key in ("groups", "label_groups", "pred_bits", "partition_counts"):
        assert np.array_equal(out[key], plain[key]), key
    assert out["partition"] == plain["partition"] and out["exact_partitions"] == plain["exact_partitions"]
    for f, v in plain_files.items():
        assert np.array_equal(np.load(d / f"{f}{Ne}.npy"), v)
    k = len(out["partition"])
    assert logs[-3 - k:-1] == plain_logs[-3 - k:-1]                  # grouping, partition_* and exact_partitions lines
    assert logs[-1].startswith("test time:")
    lab = _cuda(out["label_groups"])
    assert list(out["sweep"]) == sweep
    for t, v in out["sweep"].items():
        want = partition_metrics_from_counts(partition_counts(hunk_clusters(pt, nh, t)[0], lab, nh).cpu().numpy())
        assert v == want, t
    rec = hunk_linkage(pt, nh)
    merges, heights, nmerges = (x.cpu().numpy() for x in rec)
    saved = np.load(d / f"C_linkage{Ne}.npz")
    _same_record((saved["merges"], saved["heights"], saved["nmerges"]), (merges, heights, nmerges))
    _same_record(out["linkage"], (merges, heights, nmerges))
    target = out["partition_counts"][:, 5].astype(np.int32)
    at_k = oracle_cut(merges, heights, nmerges, test.nh[:n].astype(np.int32), target=target)[0][0]
    want = partition_metrics_from_counts(partition_counts(_cuda(at_k), lab, nh).cpu().numpy())
    assert out["sweep_labelled_k"] == want
    start = len(logs) - 4 - k - len(sweep)
    assert logs[start:start + len(sweep)] == [f"sweep threshold {t}: {v}" for t, v in out["sweep"].items()]
    assert logs[start + len(sweep)] == f"sweep labelled groups: {out['sweep_labelled_k']}"
    assert logs[start + len(sweep) + 1] == f"grouping: average linkage, threshold {thr}"
    model.engine.close()
