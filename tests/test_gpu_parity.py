"""GPU parity: the CUDA path behind the C ABI vs the CPU oracle (fp64 closed form + autograd) on
the same seeded inputs.  Tolerance: the north-star's fp32 budget, max rel err <= 1e-3, measured
as max|cuda - oracle| / max|oracle| per tensor (fp32 kernels actually land near 1e-6)."""
import numpy as np
import pytest
import torch

from hdgnn_b200.synthetic import make_commits
from oracle import hdgnn_oracle as O
from oracle import plan_numpy as PN

pytestmark = pytest.mark.gpu

TOL = 1e-3          # north-star budget
TIGHT = 1e-4        # what an all-fp32 path should achieve


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _params(variant, seed=7):
    flat = O.init_params(variant, seed=seed, dtype=torch.float64)
    g = torch.Generator().manual_seed(seed + 1)
    return flat + 0.05 * torch.randn(flat.numel(), generator=g, dtype=torch.float64)


CASES = [
    # B, Ne, Nc, variant
    (3, 9, 5, 2), (2, 33, 12, 2), (4, 40, 20, 1), (3, 37, 21, 3), (2, 33, 12, 4), (3, 64, 32, 4),
    (5, 70, 33, 2), (2, 200, 74, 2), (2, 97, 74, 4), (2, 250, 114, 2), (2, 160, 150, 2),
    # hunk tables in the per-commit global slice (Nc > 128), also under the dense-sweep flag and for variant 4
    (2, 120, 170, 2), (2, 100, 200, 4), (2, 90, 140, 1),
]


F_DEBUG, F_LEGACY, F_LABEL_BITS, F_DENSE = 2, 4, 8, 16
PATH_FLAGS = {"default": 0, "dense": F_DENSE, "legacy": F_LEGACY}


@pytest.mark.parametrize("path", ["default", "dense", "legacy"])
@pytest.mark.parametrize("B,Ne,Nc,variant", CASES)
def test_forward_backward_matches_oracle(B, Ne, Nc, variant, path):
    from hdgnn_b200.engine import Engine, DeviceBatch
    cb = make_commits(B, Ne, Nc, seed=100 + Ne, p_edge=0.1, p_short=0.5, p_noise=0.1)
    flat = _params(variant)
    plan = PN.train_step_plan(variant, flat, cb.adj, cb.x, cb.hmap, cb.L, cb.Y)
    if Ne <= 70:     # autograd oracle as an independent check of the plan at this size
        _, ce, _, grad, out = O.train_loss_and_grad(variant, flat, cb.adj, cb.x, cb.hmap, cb.L, cb.Y)
        assert relerr(plan["grad"], grad.numpy()) < 1e-9
        assert relerr(plan["logits"], out["logits"].numpy()) < 1e-10

    if path == "dense" and variant != 2:
        pytest.skip("the dense-sweep flag only changes variant 2")
    eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=F_DEBUG | PATH_FLAGS[path])
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    params = flat.float().cuda()
    probs, logits, loss, grads = eng.forward_backward(db, params, want_logits=True)
    torch.cuda.synchronize()
    if path != "legacy" and Nc <= 256 and (variant != 4 or eng.last_launch_count() <= 5):
        # the fused path ran: pack_bits, mid (entity pair layer inline), reduce -- or, with the dense entity sweeps (flag, or the
        # inline state not fitting one SM next to mid's: Ne=250 with Nc=150), pack_bits, ent_fwd, mid, ent_bwd, reduce
        want = (3,) if variant not in (2, 4) else ((5,) if path == "dense" else (3, 5))
        assert eng.last_launch_count() in want, eng.last_launch_count()
    errs = {}
    I = plan["I"]
    def ws(name, shape):
        return eng.workspace(name, shape).cpu().numpy()
    if variant in (2, 4):
        if path == "legacy" or eng.last_launch_count() >= 5:      # inline entity stage (variants 2 and 4): only RS + CS exists
            errs["RS1"] = relerr(ws("RS1", (B, Ne, 20)), I["RS1"])
        errs["S1"] = relerr(ws("S1", (B, Ne, 20)), I["RS1"] + I["CS1"])
        errs["X2"] = relerr(ws("X2", (B, Ne)), I["x2"])
    errs["NB"] = relerr(ws("NB", (B, Nc, 4)), I["nb"])
    errs["RS3"] = relerr(ws("RS3", (B, Nc, 20)), I["RS3"])
    errs["CS3F"] = relerr(ws("CS3F", (B, Nc, 20)), I["CS3"])
    errs["PR"] = relerr(ws("PR", (B, Nc, 20)), I["PR"])
    errs["PC"] = relerr(ws("PC", (B, Nc, 20)), I["PC"])
    errs["logits"] = relerr(logits.cpu().numpy(), plan["logits"])
    errs["probs"] = relerr(probs.cpu().numpy(), plan["probs"])
    errs["ce"] = relerr(loss.cpu().numpy()[0], plan["ce"])
    errs["DNB"] = relerr(ws("DNB", (B, Nc, 4)), I["dnb"])
    if variant in (2, 4):
        errs["DX2"] = relerr(ws("DX2", (B, Ne)), I["dx2"])
        errs["GE"] = relerr(ws("GE", (B, Ne, 20)), I["gE"])
    # CE gradient only (the regularisers live in the Adam kernel)
    pf = flat.numpy()
    reg = 0.001 * pf
    offs = {n: o for n, o in zip([s[0] for s in O.param_spec(variant)],
                                 np.cumsum([0] + [int(np.prod(s[2])) for s in O.param_spec(variant)])[:-1])}
    for t in ("theta1", "theta2"):
        th = pf[offs[t]:offs[t] + 2]
        reg[offs[t]:offs[t] + 2] += 0.001 * th / np.sqrt((th ** 2).sum())
    g_ce = plan["grad"] - reg
    g_cuda = grads.cpu().numpy()
    errs["grad"] = relerr(g_cuda, g_ce)
    # per-block gradient errors, relative to the block's own scale
    spec = O.param_spec(variant)
    for (name, _, shape) in spec:
        n = int(np.prod(shape)); o = offs[name]
        ref = g_ce[o:o + n]
        if np.abs(ref).max() > 0:
            errs["g_" + name] = relerr(g_cuda[o:o + n], ref)
        else:
            assert np.abs(g_cuda[o:o + n]).max() == 0, name
    bad = {k: v for k, v in errs.items() if not (v < TOL)}
    assert not bad, f"above the 1e-3 budget: {bad}\nall: {errs}"
    loose = {k: v for k, v in errs.items() if not (v < TIGHT)}
    assert not loose, f"fp32 path should be within {TIGHT}: {loose}"
    # predicted relation classes identical (argmax over the 2 channels), away from exact ties
    pc = probs.cpu().numpy(); pp = plan["probs"]
    sure = np.abs(pp[:, 1] - pp[:, 0]) > 1e-4
    assert np.array_equal((pc[:, 1] > pc[:, 0])[sure], (pp[:, 1] > pp[:, 0])[sure])
    eng.close()


@pytest.mark.parametrize("variant", [1, 2, 4])
def test_forward_only_matches_training_forward(variant):
    from hdgnn_b200.engine import Engine, DeviceBatch
    B, Ne, Nc = 3, 50, 23
    cb = make_commits(B, Ne, Nc, seed=5)
    flat = _params(variant)
    eng = Engine(Ne, Nc, variant=variant, max_batch=B)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    params = flat.float().cuda()
    p1, l1, loss1 = eng.forward(db, params)
    p2, l2, loss2, _ = eng.forward_backward(db, params, want_logits=True)
    torch.cuda.synchronize()
    if eng.last_launch_count() > 6 and variant == 4:
        # variant 4: inference runs on the fused path while the training step may still take the multi-kernel path: same numbers
        # up to fp32 summation order
        assert torch.allclose(p1, p2, atol=2e-6) and torch.allclose(l1, l2, rtol=1e-5, atol=1e-4) and torch.allclose(loss1, loss2, rtol=1e-5)
    else:
        assert torch.equal(p1, p2) and torch.equal(l1, l2) and torch.equal(loss1, loss2)
    eng.close()


@pytest.mark.parametrize("variant", [2, 4])
def test_run_to_run_bitwise_determinism(variant):
    from hdgnn_b200.engine import Engine, DeviceBatch
    B, Ne, Nc = 6, 120, 50
    cb = make_commits(B, Ne, Nc, seed=9)
    eng = Engine(Ne, Nc, variant=variant, max_batch=B)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    params = _params(variant).float().cuda()
    outs = []
    for _ in range(3):
        p, _, l, g = eng.forward_backward(db, params)
        torch.cuda.synchronize()
        outs.append((p.clone(), l.clone(), g.clone()))
    for o in outs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(outs[0], o))
    eng.close()


def test_adam_step_matches_tf_formula():
    from hdgnn_b200.engine import Engine
    variant = 2
    eng = Engine(16, 8, variant=variant, max_batch=1)
    n = eng.n_params
    rng = np.random.default_rng(3)
    p = rng.normal(scale=0.1, size=n); g = rng.normal(scale=0.01, size=n)
    m = np.zeros(n); v = np.zeros(n)
    pt = torch.tensor(p, dtype=torch.float32).cuda(); gt = torch.tensor(g, dtype=torch.float32).cuda()
    mt = torch.zeros(n, device="cuda"); vt = torch.zeros(n, device="cuda")
    step = torch.zeros(1, dtype=torch.int32, device="cuda"); reg = torch.zeros(2, device="cuda")
    offs = {s[0]: o for s, o in zip(O.param_spec(variant), np.cumsum([0] + [int(np.prod(s[2])) for s in O.param_spec(variant)])[:-1])}
    for t in range(1, 4):
        full = g + 0.001 * p
        for th in ("theta1", "theta2"):
            o = offs[th]
            full[o:o + 2] += 0.001 * p[o:o + 2] / np.sqrt((p[o:o + 2] ** 2).sum())
        lm, lp = O.reg_loss(torch.tensor(p), variant)
        p, m, v = O.tf_adam_step(p, full, m, v, t)
        eng.adam_step(pt, gt, mt, vt, step, reg_losses=reg)
        torch.cuda.synchronize()
        assert int(step.item()) == t
        assert relerr(pt.cpu().numpy(), p) < 1e-6
        assert relerr(mt.cpu().numpy(), m) < 1e-5 and relerr(vt.cpu().numpy(), v) < 5e-5   # 1-0.999f
        assert relerr(reg.cpu().numpy(), np.array([float(lm), float(lp)])) < 1e-5
    eng.close()


# host inputs of the *_host entry points: byte grids (staged by events, re-pitched on the device); label bitmaps in one pinned
# HostBatch block (one DMA, ordered by a tag the per-commit kernel polls) or in five separate pinned tensors (one DMA per
# section); label bitmaps into a dense-sweep handle, whose first kernel is ent_fwd2 (ordered by an event instead of the tag)
HOST_INPUTS = {"bytes": 0, "bits_block": F_LABEL_BITS, "bits_sections": F_LABEL_BITS, "dense_bits": F_LABEL_BITS | F_DENSE}


def test_host_entry_points_match_device_entry_points():
    _host_entry_points_match_device_entry_points("bytes")


@pytest.mark.parametrize("inputs", ["bits_block", "bits_sections", "dense_bits"])
def test_host_entry_points_match_device_entry_points_label_bits(inputs):
    _host_entry_points_match_device_entry_points(inputs)


def _host_entry_points_match_device_entry_points(inputs):
    from hdgnn_b200.engine import Engine, DeviceBatch, pack_label_bits
    from hdgnn_b200.model import HostBatch
    B, Ne, Nc, variant = 4, 50, 20, 2      # Ne, Nc not multiples of 16: exercises the pitched staging copy
    cb = make_commits(B, Ne, Nc, seed=21)
    flat = _params(variant).float()
    flags = HOST_INPUTS[inputs]
    bits = bool(flags & F_LABEL_BITS)
    eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=flags)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev, bits=bits)
    params = flat.cuda()
    probs, _, loss, grads = eng.forward_backward(db, params)
    p_ref = params.clone(); m = torch.zeros_like(params); v = torch.zeros_like(params)
    step = torch.zeros(1, dtype=torch.int32, device="cuda"); reg = torch.zeros(2, device="cuda")
    eng.adam_step(p_ref, grads, m, v, step, reg_losses=reg)
    pin = lambda a: torch.as_tensor(np.ascontiguousarray(a)).pin_memory()
    if inputs == "bits_sections":
        h = [pin(pack_label_bits(cb.adj).view(np.int32)), pin(cb.x), pin(cb.hmap), pin(cb.L), pin(pack_label_bits(cb.Y).view(np.int32))]
    elif bits:
        h = list(HostBatch(cb, bits=True).tensors())
    else:
        h = [pin(cb.adj), pin(cb.x), pin(cb.hmap), pin(cb.L), pin(cb.Y)]
    p2 = flat.cuda(); m2 = torch.zeros_like(p2); v2 = torch.zeros_like(p2)
    step2 = torch.zeros(1, dtype=torch.int32, device="cuda")
    loss3 = torch.zeros(3).pin_memory(); probs_h = torch.zeros(B, 2, eng.Ncr).pin_memory()
    eng.train_step_host(*h, p2, m2, v2, step2, loss3, probs=probs_h)
    torch.cuda.synchronize()
    assert torch.allclose(p2, p_ref, rtol=1e-6, atol=1e-9)
    assert torch.equal(probs_h, probs.cpu())
    assert abs(loss3[0].item() - loss.item()) <= 1e-6 * abs(loss.item())
    assert torch.allclose(loss3[1:], reg.cpu(), rtol=1e-6)     # different (fixed) summation orders
    # commit-sharded host entry: same gradient as the device entry, back-to-back calls alternate staging slots
    for _ in range(3):
        g2 = torch.zeros_like(grads); l2 = torch.zeros(1, device="cuda"); pr2 = torch.zeros_like(probs)
        eng.forward_backward_host(*h, flat.cuda(), g2, B, loss=l2, probs=pr2)
        torch.cuda.synchronize()
        assert torch.equal(g2, grads) and torch.equal(pr2, probs) and torch.equal(l2, loss)
    probs_i = torch.zeros(B, 2, eng.Ncr).pin_memory(); li = torch.zeros(1).pin_memory()
    eng.infer_host(*h, flat.cuda(), probs_i, li)
    torch.cuda.synchronize()
    assert torch.equal(probs_i, probs.cpu()) and abs(li.item() - loss.item()) <= 1e-6 * abs(loss.item())
    eng.close()


def test_argument_validation():
    from hdgnn_b200.engine import Engine, DeviceBatch
    from hdgnn_b200._lib import HdgnnError
    with pytest.raises(HdgnnError):
        Engine(600, 10)
    with pytest.raises((HdgnnError, ValueError)):
        Engine(10, 10, variant=7)
    eng = Engine(20, 10, max_batch=2)
    cb = make_commits(3, 20, 10, seed=1)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    with pytest.raises(HdgnnError):
        eng.forward(db, torch.zeros(eng.n_params, device="cuda"))     # B > max_batch
    eng.close()


@pytest.mark.parametrize("variant", [1, 2, 4])
def test_fused_train_step_matches_separate_calls(variant):
    """hdgnn_train_step (one call) == hdgnn_forward_backward + hdgnn_adam_step, and both follow the oracle's
    TF-Adam trajectory for three steps."""
    from hdgnn_b200.engine import Engine, DeviceBatch
    B, Ne, Nc = 5, 45, 19
    cb = make_commits(B, Ne, Nc, seed=33, p_short=0.5)
    flat = _params(variant)
    eng = Engine(Ne, Nc, variant=variant, max_batch=B)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    pa = flat.float().cuda(); ma = torch.zeros_like(pa); va = torch.zeros_like(pa)
    pb = flat.float().cuda(); mb = torch.zeros_like(pb); vb = torch.zeros_like(pb)
    sa = torch.zeros(1, dtype=torch.int32, device="cuda"); sb = torch.zeros(1, dtype=torch.int32, device="cuda")
    loss3 = torch.zeros(3, device="cuda"); reg = torch.zeros(2, device="cuda")
    p_ref = flat.clone(); m_ref = torch.zeros_like(flat); v_ref = torch.zeros_like(flat)
    for t in range(1, 4):
        eng.train_step(db, pa, ma, va, sa, loss3)
        _, _, loss, g = eng.forward_backward(db, pb)
        eng.adam_step(pb, g, mb, vb, sb, reg_losses=reg)
        _, ce, _, grad, _ = O.train_loss_and_grad(variant, p_ref, cb.adj, cb.x, cb.hmap, cb.L, cb.Y)
        p_ref, m_ref, v_ref = O.tf_adam_step(p_ref, grad, m_ref, v_ref, t)
        torch.cuda.synchronize()
        assert int(sa.item()) == t and int(sb.item()) == t
        assert torch.allclose(pa, pb, rtol=1e-6, atol=1e-9)
        assert abs(loss3[0].item() - loss.item()) <= 1e-6 * abs(loss.item())
        assert torch.allclose(loss3[1:], reg, rtol=1e-6)
        assert relerr(pa.cpu().numpy(), p_ref.numpy()) < TIGHT
        assert abs(loss3[0].item() - float(ce)) < TIGHT * float(ce)
    eng.close()


def _edge_batches():
    """Inputs at the edges of the domain (utils2.py:111-137): index files with 0, 1 or 2 lines, every line 'null',
    every entity in ONE hunk, empty and complete adjacency / label grids, zero node attributes."""
    Ne, Nc, B = 40, 12, 8
    cb = make_commits(B, Ne, Nc, seed=77, p_edge=0.15, p_short=0.0, p_noise=0.1)
    cb.L[0], cb.L[1], cb.L[2], cb.L[3] = 0, 1, 2, 3
    cb.hmap[4, :] = -1                       # all lines 'null' (or cut by the Nc rule): nothing is pooled
    cb.hmap[5, :] = 7                        # every entity in one hunk
    cb.adj[6] = 0; cb.Y[6] = 0               # no entity edge, no related hunk pair
    cb.adj[7] = 1; cb.Y[7] = 1               # complete graphs
    idx = np.arange(Ne); cb.adj[7, idx, idx] = 0
    cidx = np.arange(Nc); cb.Y[7, cidx, cidx] = 0
    cb.x[3] = 0.0
    return cb, Ne, Nc, B


@pytest.mark.parametrize("path", ["default", "dense", "legacy"])
@pytest.mark.parametrize("variant", [1, 2, 4])
def test_domain_edge_cases_match_oracle(variant, path):
    from hdgnn_b200.engine import Engine, DeviceBatch
    cb, Ne, Nc, B = _edge_batches()
    flat = _params(variant)
    plan = PN.train_step_plan(variant, flat, cb.adj, cb.x, cb.hmap, cb.L, cb.Y)
    _, ce, _, grad, out = O.train_loss_and_grad(variant, flat, cb.adj, cb.x, cb.hmap, cb.L, cb.Y)
    assert relerr(plan["grad"], grad.numpy()) < 1e-9 and relerr(plan["probs"], out["probs"].numpy()) < 1e-10
    if path == "dense" and variant != 2:
        pytest.skip("the dense-sweep flag only changes variant 2")
    eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=PATH_FLAGS[path])
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    params = flat.float().cuda()
    probs, logits, loss, grads = eng.forward_backward(db, params, want_logits=True)
    torch.cuda.synchronize()
    assert torch.isfinite(probs).all() and torch.isfinite(grads).all()
    pf = flat.numpy()
    reg = 0.001 * pf
    names = [s[0] for s in O.param_spec(variant)]
    offs = dict(zip(names, np.cumsum([0] + [int(np.prod(s[2])) for s in O.param_spec(variant)])[:-1]))
    for t in ("theta1", "theta2"):
        th = pf[offs[t]:offs[t] + 2]
        reg[offs[t]:offs[t] + 2] += 0.001 * th / np.sqrt((th ** 2).sum())
    errs = {"probs": relerr(probs.cpu().numpy(), plan["probs"]), "logits": relerr(logits.cpu().numpy(), plan["logits"]),
            "ce": relerr(loss.cpu().numpy()[0], plan["ce"]), "grad": relerr(grads.cpu().numpy(), plan["grad"] - reg)}
    # per commit, so that a wrong degenerate commit cannot hide behind the others
    for b in range(B):
        errs[f"probs[{b}]"] = relerr(probs[b].cpu().numpy(), plan["probs"][b])
    assert all(v < TIGHT for v in errs.values()), errs
    # a single-commit batch through the same engine
    one = DeviceBatch.from_numpy(cb.adj[1:2], cb.x[1:2], cb.hmap[1:2], cb.L[1:2], cb.Y[1:2], eng.tdev)
    p1, _, _, _ = eng.forward_backward(one, params)
    torch.cuda.synchronize()
    assert relerr(p1.cpu().numpy(), plan["probs"][1:2]) < TIGHT
    eng.close()


@pytest.mark.parametrize("Ne,Nc", [(2, 2), (3, 2), (2, 5)])
def test_smallest_grids(Ne, Nc):
    from hdgnn_b200.engine import Engine, DeviceBatch
    cb = make_commits(3, Ne, Nc, seed=5, p_edge=0.5, p_short=0.0, p_noise=0.5)
    flat = _params(2)
    plan = PN.train_step_plan(2, flat, cb.adj, cb.x, cb.hmap, cb.L, cb.Y)
    eng = Engine(Ne, Nc, variant=2, max_batch=3)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    probs, _, loss, grads = eng.forward_backward(db, flat.float().cuda())
    torch.cuda.synchronize()
    assert relerr(probs.cpu().numpy(), plan["probs"]) < TIGHT and relerr(loss.cpu().numpy()[0], plan["ce"]) < TIGHT
    eng.close()


@pytest.mark.parametrize("attr", ["many_integers", "continuous", "two_values", "constant"])
@pytest.mark.parametrize("B,Ne,Nc,p_edge", [(3, 70, 33, 0.1), (2, 200, 74, 0.05), (2, 130, 40, 0.6), (2, 120, 170, 0.1), (1, 512, 256, 0.05)])
def test_entity_stage_attribute_alphabets(B, Ne, Nc, p_edge, attr):
    """The inline entity pair layer picks its form per commit from the node attributes (utils2.py:35: x_i = A_ii): class
    tables for at most 16 distinct values, sorted prefix sums + edge walk otherwise.  Both against the oracle, including
    dense graphs (the edge walk's worst case) and degenerate alphabets; the last two shapes keep the hunk tables (and the
    class tables' neighbour counts) in global memory."""
    from hdgnn_b200.engine import Engine, DeviceBatch
    cb = make_commits(B, Ne, Nc, seed=500 + Ne, p_edge=p_edge, p_short=0.5)
    rng = np.random.default_rng(Ne)
    if attr == "many_integers":
        cb.x[:] = rng.integers(0, 40, size=cb.x.shape)
    elif attr == "continuous":
        cb.x[:] = rng.normal(scale=2.0, size=cb.x.shape)
        cb.x[0, :5] = cb.x[0, 5]                       # ties in the sort
    elif attr == "two_values":
        cb.x[:] = rng.integers(0, 2, size=cb.x.shape)
    else:
        cb.x[:] = 3.0
    flat = _params(2)
    plan = PN.train_step_plan(2, flat, cb.adj, cb.x, cb.hmap, cb.L, cb.Y)
    eng = Engine(Ne, Nc, variant=2, max_batch=B, flags=F_DEBUG)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev)
    probs, logits, loss, grads = eng.forward_backward(db, flat.float().cuda(), want_logits=True)
    torch.cuda.synchronize()
    assert eng.last_launch_count() == 3                # pack_bits, mid (entity stage inline), reduce
    I = plan["I"]
    pf = flat.numpy()
    reg = 0.001 * pf
    names = [s[0] for s in O.param_spec(2)]
    offs = dict(zip(names, np.cumsum([0] + [int(np.prod(s[2])) for s in O.param_spec(2)])[:-1]))
    for t in ("theta1", "theta2"):
        th = pf[offs[t]:offs[t] + 2]
        reg[offs[t]:offs[t] + 2] += 0.001 * th / np.sqrt((th ** 2).sum())
    g_ce, g_cuda = plan["grad"] - reg, grads.cpu().numpy()
    errs = {"S1": relerr(eng.workspace("S1", (B, Ne, 20)).cpu().numpy(), I["RS1"] + I["CS1"]),
            "X2": relerr(eng.workspace("X2", (B, Ne)).cpu().numpy(), I["x2"]),
            "GE": relerr(eng.workspace("GE", (B, Ne, 20)).cpu().numpy(), I["gE"]),
            "logits": relerr(logits.cpu().numpy(), plan["logits"]), "ce": relerr(loss.cpu().numpy()[0], plan["ce"]),
            "grad": relerr(g_cuda, g_ce)}
    for name in ("ent_w1", "ent_b1"):
        n = 80 if name == "ent_w1" else 20
        o = offs[name]
        errs["g_" + name] = relerr(g_cuda[o:o + n], g_ce[o:o + n])
    assert all(v < TIGHT for v in errs.values()), errs
    eng.close()
