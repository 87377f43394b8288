"""GPU tests of the untangling output: the predicted-relation bitmap the relation head writes (hdgnn_set_predictions) on every
form of the per-commit kernel and on the multi-kernel path, the hunk groups kernel (hdgnn_hunk_groups) against scipy, host-fed
inference without probabilities, and graph2graph.untangle end to end.  Every comparison is integer and exact."""
import numpy as np
import pytest
import torch
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

from hdgnn_b200 import _lib
from hdgnn_b200.engine import (Engine, DeviceBatch, F_LABEL_BITS, F_LEGACY, bit_words, hunk_groups, pack_label_bits)
from hdgnn_b200.synthetic import make_commits

pytestmark = pytest.mark.gpu


def _argmax_bits(probs: torch.Tensor, Nc: int) -> np.ndarray:
    """pack_label_bits of [p1 > p0] (np.argmax, a tie is class 0), pairs in the order p(s,t) = s(Nc-1)+t-[t>s]."""
    p = probs.cpu().numpy()
    B = p.shape[0]
    grid = np.zeros((B, Nc, Nc), dtype=np.uint8)
    grid[:, ~np.eye(Nc, dtype=bool)] = p[:, 1] > p[:, 0]
    return pack_label_bits(grid)


def _centred_params(eng, db, variant, seed=5):
    """Random weights with the head bias moved to the median logit difference, so both classes get predicted."""
    g = torch.Generator().manual_seed(seed)
    params = (0.3 * torch.randn(eng.n_params, generator=g)).cuda()
    _, logits, _ = eng.forward(db, params, want_logits=True)
    off = _lib.lib.hdgnn_param_offset(variant, b"scr_b2")
    params[off + 1] -= (logits[:, 1] - logits[:, 0]).median()
    return params


def _garbage(shape):
    """An int32 buffer of 0xFF bytes: every bit the kernel leaves alone stays set."""
    return torch.full(shape, -1, dtype=torch.int32, device="cuda")


# (Ne, Nc, variant, flags, HDGNN_CLUSTER): the cluster form (v2 up to 128 hunks, B below one wave), the same with one CTA per
# commit, the global-slice tables (170 hunks), the forward-only 16-segment instantiation (300 hunks), variant 4 inside the
# per-commit kernel, the multi-kernel path forced (v2, v4), and variant 4 above 256 hunks (multi-kernel forward)
FORMS = [(60, 33, 2, 0, "1"), (200, 74, 2, 0, "1"), (60, 33, 2, 0, "0"), (200, 74, 2, 0, "0"), (120, 170, 2, 0, "1"),
         (90, 300, 1, 0, "1"), (200, 74, 4, 0, "1"), (200, 74, 2, F_LEGACY, "1"), (200, 74, 4, F_LEGACY, "1"),
         (90, 300, 4, 0, "1")]


@pytest.mark.parametrize("Ne,Nc,variant,flags,cluster", FORMS)
def test_predicted_bitmap_is_argmax_of_probs(monkeypatch, Ne, Nc, variant, flags, cluster):
    monkeypatch.setenv("HDGNN_CLUSTER", cluster)
    B = 5
    cb = make_commits(B, Ne, Nc, seed=77 + Nc, p_short=0.4, p_noise=0.3)
    eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=flags)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    params = _centred_params(eng, db, variant)
    pred = _garbage((B, Nc, bit_words(Nc)))
    eng.set_predictions(pred)
    probs, _, _ = eng.forward(db, params, want_logits=False)
    torch.cuda.synchronize()
    ref = _argmax_bits(probs, Nc)
    got = pred.cpu().numpy().view(np.uint32)
    assert np.array_equal(got, ref)
    ones = int(np.unpackbits(ref.view(np.uint8)).sum())
    assert 0 < ones < B * Nc * (Nc - 1)                  # both predictions occur
    # predictions off: the buffer is left alone
    eng.set_predictions(None)
    keep = pred.clone()
    eng.forward(db, params * 1.5, want_logits=False)
    torch.cuda.synchronize()
    assert torch.equal(pred, keep)
    eng.close()


@pytest.mark.parametrize("flags", [0, F_LEGACY])
def test_training_step_writes_the_argmax_of_its_probs(flags):
    """A training call writes the predictions of the probabilities the same step writes (glide, B = 100), in the per-commit
    kernel and in the training instantiation of the multi-kernel relation head."""
    Ne, Nc, B = 200, 74, 100
    cb = make_commits(B, Ne, Nc, seed=31, p_short=0.3, p_noise=0.3)
    eng = Engine(Ne, Nc, variant=2, max_batch=B, flags=flags)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    params = _centred_params(eng, db, 2, seed=9)
    m, v = torch.zeros_like(params), torch.zeros_like(params)
    step = torch.zeros(1, dtype=torch.int32, device="cuda")
    loss3 = torch.zeros(3, dtype=torch.float32, device="cuda")
    probs = torch.empty(B, 2, Nc * (Nc - 1), dtype=torch.float32, device="cuda")
    pred = _garbage((B, Nc, bit_words(Nc)))
    eng.set_predictions(pred)
    eng.train_step(db, params, m, v, step, loss3, probs=probs)
    torch.cuda.synchronize()
    assert np.array_equal(pred.cpu().numpy().view(np.uint32), _argmax_bits(probs, Nc))
    eng.set_predictions(None)
    keep = pred.clone()
    eng.train_step(db, params, m, v, step, loss3, probs=probs)
    torch.cuda.synchronize()
    assert torch.equal(pred, keep)
    eng.close()


# ---- hunk groups ------------------------------------------------------------------------------------------------
def _scipy_groups(A: np.ndarray):
    """(n, n) {0,1} -> (groups labelled by the smallest index of the weak component, count)."""
    n = A.shape[0]
    A = A.copy()
    np.fill_diagonal(A, 0)
    k, lab = connected_components(csr_matrix(A), directed=True, connection="weak")
    first = np.full(k, n, dtype=np.int64)
    np.minimum.at(first, lab, np.arange(n))
    return first[lab].astype(np.int32), k


def _graphs(n, rng):
    """(kinds, n, n) uint8 adjacency of the cases: empty, complete, sparse random directed, one backward edge, planted blocks
    under a random permutation, a path through every hunk in random order (directions random)."""
    out = [np.zeros((n, n), np.uint8), np.ones((n, n), np.uint8)]
    for p in (1.0 / n, 2.0 / n, 0.05):
        out.append((rng.random((n, n)) < p).astype(np.uint8))
    one = np.zeros((n, n), np.uint8)
    one[n - 1, 0] = 1                                    # a single edge, stored in one direction only
    out.append(one)
    perm = rng.permutation(n)
    blocks = np.zeros((n, n), np.uint8)
    cuts = np.sort(rng.choice(np.arange(1, n), size=min(5, n - 1), replace=False))
    for blk in np.split(perm, cuts):
        for a, b in zip(blk[:-1], blk[1:]):              # a chain keeps every block connected...
            if rng.random() < 0.5:
                blocks[a, b] = 1
            else:
                blocks[b, a] = 1
        for _ in range(len(blk)):                        # ...plus random edges inside it
            a, b = rng.choice(blk, 2)
            blocks[a, b] = 1
    out.append(blocks)
    path = np.zeros((n, n), np.uint8)
    order = rng.permutation(n)
    for a, b in zip(order[:-1], order[1:]):
        if rng.random() < 0.5:
            path[a, b] = 1
        else:
            path[b, a] = 1
    out.append(path)
    return np.stack(out)


def _with_garbage(A: np.ndarray, rng) -> np.ndarray:
    """Label bitmap of A with random diagonal bits and random padding bits (columns >= n, padding words)."""
    B, n, _ = A.shape
    wp = bit_words(n)
    wide = (rng.random((B, n, wp * 32)) < 0.5).astype(np.uint8)
    wide[:, :, :n] = A
    wide[:, np.arange(n), np.arange(n)] = rng.random((B, n)) < 0.5
    return np.ascontiguousarray(np.packbits(wide, axis=-1, bitorder="little")).view("<u4").reshape(B, n, wp)


@pytest.mark.parametrize("n", [2, 31, 32, 33, 74, 150, 256, 300, 512])
def test_hunk_groups_equal_scipy_weak_components(n):
    rng = np.random.default_rng(1000 + n)
    A = _graphs(n, rng)
    bits = torch.as_tensor(_with_garbage(A, rng).view(np.int32)).cuda()
    groups, ngroups = hunk_groups(bits)
    again, ng2 = hunk_groups(bits)
    torch.cuda.synchronize()
    assert torch.equal(groups, again) and torch.equal(ngroups, ng2)
    g, ng = groups.cpu().numpy(), ngroups.cpu().numpy()
    for k in range(A.shape[0]):
        ref, cnt = _scipy_groups(A[k])
        assert np.array_equal(g[k], ref), (n, k)
        assert int(ng[k]) == cnt, (n, k)
    assert np.array_equal(g[0], np.arange(n)) and ng[0] == n              # empty graph
    assert not g[1].any() and ng[1] == 1                                   # complete graph
    if n > 2:
        assert g[5][n - 1] == 0 and ng[5] == n - 1                         # one direction alone joins two hunks
    assert not g[-1].any() and ng[-1] == 1                                 # the path joins everything


def test_hunk_groups_of_many_commits():
    """Batches that put several commits into one CTA."""
    for n, B in ((74, 1001), (512, 400)):          # 1001: the last CTA of four-commit CTAs has idle warps
        rng = np.random.default_rng(n)
        A = (rng.random((B, n, n)) < 1.2 / n).astype(np.uint8)
        g, ng = hunk_groups(torch.as_tensor(pack_label_bits(A).view(np.int32)).cuda())
        g, ng = g.cpu().numpy(), ng.cpu().numpy()
        for k in range(0, B, 37):
            ref, cnt = _scipy_groups(A[k])
            assert np.array_equal(g[k], ref) and ng[k] == cnt


# ---- host-fed inference without probabilities ------------------------------------------------------------------
@pytest.mark.parametrize("Ne,Nc,variant", [(200, 74, 2), (90, 300, 4)])
def test_infer_host_without_probs_gives_the_device_bits_and_loss(Ne, Nc, variant):
    from hdgnn_b200.model import HostBatch
    B = 20
    cb = make_commits(B, Ne, Nc, seed=3 + Nc, p_short=0.3, p_noise=0.3)
    eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=F_LABEL_BITS)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev, bits=True)
    params = _centred_params(eng, db, variant)
    ref_bits = _garbage((B, Nc, bit_words(Nc)))
    eng.set_predictions(ref_bits)
    _, _, ref_loss = eng.forward(db, params, want_logits=False)
    hb = HostBatch(cb, bits=True)
    bits = _garbage((B, Nc, bit_words(Nc)))
    loss = torch.zeros(1, dtype=torch.float32).pin_memory()
    eng.set_predictions(bits)
    eng.infer_host(*hb.tensors(), params, None, loss)
    torch.cuda.synchronize()
    eng.set_predictions(None)
    assert torch.equal(bits, ref_bits)
    assert torch.equal(loss, ref_loss.cpu())
    eng.close()


# ---- graph2graph.untangle end to end ---------------------------------------------------------------------------
def test_untangle_after_train(tmp_path):
    from hdgnn_b200.model import graph2graph
    from hdgnn_b200.utils2 import write_dataset, read_compact, split_half
    Ne, Nc, N, MB = 12, 5, 16, 4
    cb = make_commits(N, Ne, Nc, seed=8, p_edge=0.2, p_short=0.4, p_noise=0.2)
    write_dataset(cb, "toy", 2, root=str(tmp_path))
    _, test = split_half(read_compact("toy", 2, Ne, Nc, root=str(tmp_path)))
    model = graph2graph(None, Ne=Ne, Nc=Nc, Mini_batch=MB, epoch=3, Step=2, Repo="toy", variant=2, seed=11,
                        checkpoint_dir=str(tmp_path / "ck"))
    model.train(None, root=str(tmp_path), log=lambda s: None)
    _, probs = model.test(None, root=str(tmp_path), log=lambda s: None)
    logs = []
    out = model.untangle(None, root=str(tmp_path), log=logs.append)
    assert any(l.startswith(" [*] Load SUCCESS") for l in logs)
    assert logs[-2].startswith("exact_partitions: ") and logs[-1].startswith("test time:")
    d = tmp_path / "outputSelf" / "toy" / "model_2" / "2"
    gt, gy = np.load(d / f"C_group_t{Ne}.npy"), np.load(d / f"C_group_y{Ne}.npy")
    n = test.B
    assert gt.shape == (n, Nc) and gy.shape == (n, Nc) and gt.dtype == np.int32 and gy.dtype == np.int32
    assert np.array_equal(gy, np.stack([_scipy_groups(test.Y[k])[0] for k in range(n)]))
    # the predictions are the arg-max of the probabilities test() writes for the same checkpoint
    pbits = _argmax_bits(torch.as_tensor(probs), Nc)
    assert np.array_equal(out["pred_bits"].view(np.uint32), pbits)
    ref, _ = hunk_groups(torch.as_tensor(pbits.view(np.int32)).cuda())
    assert np.array_equal(gt, ref.cpu().numpy())
    assert np.array_equal(out["groups"], gt) and np.array_equal(out["label_groups"], gy)
    assert out["exact_partitions"] == int((gt == gy).all(1).sum())
    assert logs[-2] == f"exact_partitions: {out['exact_partitions']} / {n}"
    model.engine.close()


def test_set_predictions_buffer_must_cover_the_batch():
    Ne, Nc, B = 60, 33, 5
    cb = make_commits(B, Ne, Nc, seed=2)
    eng = Engine(Ne, Nc, variant=2, max_batch=B)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    eng.set_predictions(_garbage((B - 1, Nc, bit_words(Nc))))
    with pytest.raises(AssertionError):
        eng.forward(db, torch.zeros(eng.n_params, device="cuda"))
    eng.set_predictions(None)
    eng.close()
