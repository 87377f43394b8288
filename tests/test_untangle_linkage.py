"""CPU checks of the average-linkage dendrogram: the oracle's merge record cut at a threshold (tests/linkage_oracle.py:
hunk_linkage + linkage_cut) equals its threshold clustering (hunk_clusters_one) at every recorded height and one ulp either
side, at +-inf, 0 and 1, and with NaN pairs; engine.scipy_linkage of the record is scipy's average linkage; both new entry
points refuse bad arguments before any CUDA call; main.py --sweep needs --grouping average."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.cluster.hierarchy import fcluster, linkage
from scipy.spatial.distance import squareform

from hdgnn_b200._lib import E_CUDA, E_INVALID, lib
from hdgnn_b200.engine import hunk_linkage, linkage_cut, scipy_linkage
from linkage_oracle import hunk_linkage_one, linkage_cut_one
from oracle.hunk_clusters import hunk_clusters_one, pair_index


def _p1(P1: np.ndarray) -> np.ndarray:
    """(n, n) channel-1 grid -> (n(n-1),) float32 in the relation head's pair order."""
    n = P1.shape[0]
    idx = pair_index(n)
    out = np.zeros(n * (n - 1), np.float32)
    out[idx[idx >= 0]] = P1[idx >= 0]
    return out


def _commit(rng, n, coarse=True):
    """Channel 1 of one commit: planted groups, uniform noise, or coarse values (many equal means: the tie rule decides)."""
    r = rng.random()
    if r < 0.25:
        return rng.random((n, n)).astype(np.float32)
    if r < 0.4 and coarse:
        return (rng.integers(0, 4, (n, n)) / 4).astype(np.float32)
    k = int(rng.integers(1, max(2, n // 3) + 1))
    g = rng.integers(0, k, size=n)
    same = g[:, None] == g[None, :]
    return np.where(same, rng.uniform(0.5, 1.0, (n, n)), rng.uniform(0.0, 0.5, (n, n))).astype(np.float32)


def _thresholds(heights):
    h = heights[~np.isnan(heights)].astype(np.float32)
    up, down = np.nextafter(h, np.float32(np.inf)), np.nextafter(h, np.float32(-np.inf))
    return np.unique(np.r_[h, up, down, np.float32([-np.inf, np.inf, 0.0, 1.0, 0.5])]).astype(np.float32)


def test_cut_of_the_linkage_equals_the_threshold_clustering():
    rng = np.random.default_rng(77)
    commits, short, cuts = 0, 0, 0
    for case in range(300):
        n = int(rng.integers(2, 25))
        m = int(rng.integers(0, n + 1)) if case % 5 == 0 else n
        P1 = _commit(rng, n)
        if case % 7 == 0 and m >= 3:                       # NaN pairs: both directions keep two hunks apart for good
            for _ in range(int(rng.integers(1, 3))):
                s, t = rng.choice(m, 2, replace=False)
                P1[s, t] = P1[t, s] = np.nan
        p1 = _p1(P1)
        merges, heights, nm = hunk_linkage_one(p1, n, m)
        assert 0 <= nm <= max(m - 1, 0)
        assert (merges[nm:] == -1).all() and np.isnan(heights[nm:]).all()
        assert (merges[:nm, 0] < merges[:nm, 1]).all() and not np.isnan(heights[:nm]).any()
        short += nm < max(m - 1, 0)
        for t in _thresholds(heights):
            want = hunk_clusters_one(p1, n, m, t)
            got = linkage_cut_one(merges, heights, nm, n, m, threshold=t)
            assert np.array_equal(got[0], want[0]) and got[1] == want[1], (case, n, m, t)
            cuts += 1
        commits += 1
    assert short >= 10 and cuts > 5000


def test_heights_store_minus_zero_as_plus_zero_and_merge_infinities():
    P1 = np.array([[0, -0.0, -np.inf], [-0.0, 0, -np.inf], [-np.inf, -np.inf, 0]], np.float32)
    merges, heights, nm = hunk_linkage_one(_p1(P1), 3, 3)
    assert nm == 2 and merges[:2].tolist() == [[0, 1], [0, 2]]
    assert heights[0] == 0 and not np.signbit(heights[0])             # -0 is stored as +0
    assert heights[1] == -np.inf                                      # recorded like any other mean
    for t, ng in ((-np.inf, 2), (np.float32(-1e-45), 2), (0.0, 3)):
        assert linkage_cut_one(merges, heights, nm, 3, 3, threshold=t)[1] == ng
        assert hunk_clusters_one(_p1(P1), 3, 3, t)[1] == ng


def test_group_count_cut():
    rng = np.random.default_rng(3)
    n = 12
    p1 = _p1(_commit(rng, n))
    merges, heights, nm = hunk_linkage_one(p1, n, 9)
    for k in range(-2, 13):
        g, ng = linkage_cut_one(merges, heights, nm, n, 9, target=k)
        assert ng == n - min(nm, max(0, 9 - max(k, 1)))
        assert len(set(g[:9].tolist())) == min(9, max(k, 1)) and np.array_equal(g[9:], np.arange(9, n))


def test_inconsistent_records_give_minus_one():
    rng = np.random.default_rng(4)
    n = 10
    merges, heights, nm = hunk_linkage_one(_p1(_commit(rng, n)), n, n)
    assert nm == n - 1
    bad = []
    for change in ("a>=c", "c twice", "a absorbed", "too many", "negative"):
        mg, k = merges.copy(), nm
        if change == "a>=c":
            mg[3] = mg[3, ::-1]
        elif change == "c twice":
            mg[5, 1] = mg[2, 1]
        elif change == "a absorbed":
            mg[6, 0] = mg[1, 1]
        elif change == "too many":
            k = n
        else:
            k = -1
        bad.append(linkage_cut_one(mg, heights, k, n, n, threshold=0.5))
    assert all((g == -1).all() and ng == -1 for g, ng in bad)
    assert linkage_cut_one(merges, heights, nm, n, n + 1, threshold=0.5)[1] == -1


def _smallest_index_labels(lab: np.ndarray) -> np.ndarray:
    first = {}
    for i, v in enumerate(lab):
        first.setdefault(v, i)
    return np.array([first[v] for v in lab], np.int32)


def _members(Z, m):
    sets = [frozenset([i]) for i in range(m)]
    rows = []
    for a, c, _, size in Z:
        a, c = sets[int(a)], sets[int(c)]
        sets.append(a | c)
        assert len(a | c) == size
        rows.append(frozenset([a, c]))
    return rows


def test_scipy_linkage_of_the_record_is_scipys_average_linkage():
    rng = np.random.default_rng(2025)
    compared, rejected = 0, 0
    while compared < 80:
        n = int(rng.integers(2, 41))
        P1 = _commit(rng, n, coarse=False)            # equal means are ordered by the tie rule here, by scipy's own there
        thr = float(rng.uniform(0.3, 0.7))
        w = np.fmax(P1, P1.T).astype(np.float64)
        np.fill_diagonal(w, 1.0)
        Zs = linkage(squareform(1.0 - w, checks=False), "average")
        h = np.sort(Zs[:, 2])
        # the same rule as the oracle's comparison with scipy: fp32 sums against fp64, so only decisions 1e-5 apart count
        if (np.diff(h) <= 1e-5).any() or (np.abs(h - (1.0 - thr)) <= 1e-5).any():
            rejected += 1
            continue
        merges, heights, nm = hunk_linkage_one(_p1(P1), n, n)
        Z = scipy_linkage(merges[None], heights[None], np.int32([nm]))[0]
        assert Z.shape == Zs.shape
        assert _members(Z, n) == _members(Zs, n)                     # the same clusters joined at every row
        assert np.abs(Z[:, 2] - Zs[:, 2]).max(initial=0) <= 1e-5
        cut = linkage_cut_one(merges, heights, nm, n, n, threshold=thr)[0]
        assert np.array_equal(_smallest_index_labels(fcluster(Z, 1.0 - thr, "distance")), cut)
        compared += 1
    assert rejected < 20


def test_scipy_linkage_refuses_a_sequence_stopped_by_nan():
    P1 = np.full((4, 4), 0.9, np.float32)
    P1[0, 1] = P1[1, 0] = np.nan
    merges, heights, nm = hunk_linkage_one(_p1(P1), 4, 4)
    assert nm == 2
    with pytest.raises(ValueError):
        scipy_linkage(merges[None], heights[None], np.int32([nm]))
    with pytest.raises(ValueError):
        scipy_linkage(merges[None], heights[None], np.int32([-1]))
    assert scipy_linkage(merges[None], heights[None], np.int32([0]), nh=[1])[0].shape == (0, 4)


# ---- arguments of the two entry points, before any CUDA call --------------------------------------------------------------
def P(addr):
    return C.c_void_p(addr)


NAN = float("nan")
THR = (C.c_float * 65)(*([0.5] * 65))
THR_NAN = (C.c_float * 3)(0.5, NAN, 0.2)
TABLE = {
    "hdgnn_hunk_linkage": (
        "B n probs nh merges heights nmerges work",
        (1, 74, P(0x10000), P(0x20000), P(0x30000), P(0x40000), P(0x50000), P(0x60000)),
        [dict(B=0), dict(n=1), dict(n=513), dict(probs=None), dict(merges=None), dict(heights=None), dict(nmerges=None),
         dict(probs=P(0x10002)), dict(nh=P(0x20001)), dict(merges=P(0x30002)), dict(heights=P(0x40003)),
         dict(nmerges=P(0x50001)), dict(work=P(0x60002), n=300),
         dict(work=None, n=300)]),                  # above n = 169 the tables need the workspace
    "hdgnn_linkage_cut": (
        "B n merges heights nmerges nh K thresholds_host target groups ngroups",
        (1, 74, P(0x10000), P(0x20000), P(0x30000), P(0x40000), 3, THR, None, P(0x60000), P(0x70000)),
        [dict(B=0), dict(n=1), dict(n=513), dict(K=0), dict(K=65), dict(K=-1),
         dict(thresholds_host=THR_NAN), dict(thresholds_host=None),                                  # neither
         dict(target=P(0x50000)),                                                                   # both
         dict(target=P(0x50000), thresholds_host=None, K=2),                                         # K = 1 with target
         dict(merges=None), dict(heights=None), dict(nmerges=None), dict(groups=None),
         dict(merges=P(0x10002)), dict(heights=P(0x20001)), dict(nmerges=P(0x30003)), dict(nh=P(0x40002)),
         dict(target=P(0x50002), thresholds_host=None, K=1), dict(groups=P(0x60001)), dict(ngroups=P(0x70002)),
         dict(thresholds_host=P(C.addressof(THR) + 2))]),
}
VALID_TOO = {"hdgnn_hunk_linkage": [dict(nh=None, work=None), dict(n=512)],
             "hdgnn_linkage_cut": [dict(nh=None, ngroups=None), dict(K=64),
                                   dict(thresholds_host=None, target=P(0x50000), K=1)]}


def _args(names, valid, change):
    names = names.split()
    assert set(change) <= set(names), change
    return [change.get(k, v) for k, v in zip(names, valid)]


@pytest.mark.parametrize("fn", sorted(TABLE))
def test_linkage_entry_points_validate_arguments_without_a_gpu(fn):
    names, valid, bad = TABLE[fn]
    for change in bad:
        assert getattr(lib, fn)(*_args(names, valid, change), None) == E_INVALID, change
        msg = lib.hdgnn_last_error(None).decode()
        assert msg.startswith(fn + ": ") and next(iter(change)) in msg[len(fn) + 2:], (change, msg)
    if not torch.cuda.is_available():                # fake pointers must never reach a real device
        for change in [{}] + VALID_TOO[fn]:
            assert getattr(lib, fn)(*_args(names, valid, change), None) == E_CUDA, change
            assert lib.hdgnn_last_error(None).decode().startswith(fn + ": ")


def test_wrappers_check_shapes_and_modes_before_the_cuda_check():
    B, n = 2, 30
    probs, nh = torch.zeros(B, 2, n * (n - 1)), torch.zeros(B, dtype=torch.int32)
    merges, heights = torch.zeros(B, n - 1, 2, dtype=torch.int32), torch.zeros(B, n - 1)
    for wrong in (lambda: hunk_linkage(probs[:, :, 1:]), lambda: hunk_linkage(probs, nh[:1]),
                  lambda: linkage_cut(merges, heights, nh, thresholds=[0.5], target=nh),     # both
                  lambda: linkage_cut(merges, heights, nh),                                  # neither
                  lambda: linkage_cut(merges, heights[:, 1:], nh, thresholds=[0.5]),
                  lambda: linkage_cut(merges, heights, nh[:1], thresholds=[0.5]),
                  lambda: linkage_cut(merges, heights, nh, target=nh[:1])):
        with pytest.raises(ValueError):
            wrong()
    for right in (lambda: hunk_linkage(probs, nh), lambda: linkage_cut(merges, heights, nh, nh, thresholds=[0.5, 0.2]),
                  lambda: linkage_cut(merges, heights, nh, target=nh)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            right()


@pytest.mark.parametrize("argv", [["--Type", "untangle", "--sweep", "0.3,0.4"],
                                  ["--Type", "test", "--grouping", "average", "--sweep", "0.3"],
                                  ["--Type", "untangle", "--grouping", "average", "--sweep", "0.3,nan"],
                                  ["--Type", "untangle", "--grouping", "average", "--sweep", "0.3,x"]])
def test_main_refuses_sweep_outside_untangle_average(argv, tmp_path, capsys):
    import main
    with pytest.raises(SystemExit) as e:
        main.main(argv + ["--root", str(tmp_path)])
    assert e.value.code == 2 and "--sweep" in capsys.readouterr().err
