"""The bit-packed wire format of the *_host entry points (HDGNN_F_LABEL_BITS): same kernels, same bitmaps, so a training
run fed with host bitmaps is BITWISE identical to one fed with byte grids (which the device packs itself) -- on the fused
path and on the multi-kernel path alike."""
import numpy as np
import pytest
import torch

from hdgnn_b200.synthetic import make_commits

F_LEGACY = 4

# (variant, Ne, Nc, B, extra flags): the fused path; HDGNN_F_LEGACY (the multi-kernel path) at variants 2 and 4; training
# above 256 hunks, which runs on the multi-kernel path while its forward-only step stays fused
WIRE_CASES = [(2, 48, 20, 5, 0), (2, 200, 74, 12, 0), (1, 33, 9, 4, 0), (3, 64, 40, 3, 0), (2, 250, 150, 3, 0),
              (2, 200, 74, 12, F_LEGACY), (4, 200, 74, 6, F_LEGACY), (2, 48, 300, 3, 0)]


def test_pack_label_bits_layout():
    from hdgnn_b200.engine import pack_label_bits, bit_words
    rng = np.random.default_rng(0)
    for n in (5, 32, 33, 74, 200, 257):
        lab = (rng.random((2, n, n)) < 0.3).astype(np.uint8)
        lab[:, np.arange(n), np.arange(n)] = 1                       # the diagonal must come out as zero
        w = pack_label_bits(lab)
        wp = bit_words(n)
        assert w.shape == (2, n, wp) and w.dtype == np.dtype("<u4") and wp % 4 == 0 and wp * 32 >= n
        cols = ((w[:, :, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(2, n, wp * 32)
        want = lab.copy(); want[:, np.arange(n), np.arange(n)] = 0
        assert np.array_equal(cols[:, :, :n], want) and not cols[:, :, n:].any()


@pytest.mark.gpu
@pytest.mark.parametrize("variant,Ne,Nc,B,extra", WIRE_CASES,
                         ids=["-".join(map(str, c[:4])) + ("-legacy" if c[4] else "") for c in WIRE_CASES])
def test_host_bits_training_is_bitwise_identical_to_byte_grids(variant, Ne, Nc, B, extra):
    from hdgnn_b200.engine import Engine, F_LABEL_BITS
    from hdgnn_b200.model import HostBatch, truncated_normal_init
    res = []
    for flags in (0, F_LABEL_BITS):
        eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=flags | extra)
        params = truncated_normal_init(variant, 3).cuda()
        m = torch.zeros_like(params); v = torch.zeros_like(params)
        step = torch.zeros(1, dtype=torch.int32, device="cuda")
        loss3 = torch.zeros(3).pin_memory()
        probs = torch.zeros(B, 2, Nc * (Nc - 1), device="cuda")
        losses = []
        for t in range(3):
            hb = HostBatch(make_commits(B, Ne, Nc, seed=40 + t), bits=bool(flags))
            eng.train_step_host(*hb.tensors(), params, m, v, step, loss3, probs=probs)
            torch.cuda.synchronize()
            losses.append(loss3.clone().numpy())
        launches = eng.last_launch_count()
        # inference through the same wire format
        ph = torch.zeros(B, 2, Nc * (Nc - 1)).pin_memory(); lh = torch.zeros(1).pin_memory()
        eng.infer_host(*hb.tensors(), params, ph, lh)
        torch.cuda.synchronize()
        res.append((params.cpu().numpy(), probs.cpu().numpy(), np.array(losses), ph.numpy().copy(), lh.numpy().copy(), launches, hb.nbytes()))
        eng.close()
    a, b = res
    for k in range(5):
        assert np.array_equal(a[k], b[k]), k
    assert b[5] < a[5]                  # no pack_bits / re-pitch kernels
    assert b[6] < a[6]                  # and fewer host->device bytes (1/8 for the label grids)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [7, 74, 200, 257, 512])
def test_device_packer_equals_host_packer(n):
    from hdgnn_b200.engine import pack_label_bits, pack_label_bits_device, label_pitch
    rng = np.random.default_rng(n)
    lab = (rng.random((3, n, n)) < 0.2).astype(np.uint8)
    g = torch.zeros(3, n, label_pitch(n), dtype=torch.uint8, device="cuda")
    g[:, :, :n] = torch.as_tensor(lab).cuda()
    assert np.array_equal(pack_label_bits_device(g).cpu().numpy().view(np.uint32), pack_label_bits(lab))


@pytest.mark.gpu
def test_label_bits_device_entry_points_bitwise():
    """Device-resident bitmaps through hdgnn_train_step / hdgnn_forward == byte grids, on the fused path and (HDGNN_F_LEGACY)
    on the multi-kernel path."""
    from hdgnn_b200.engine import Engine, DeviceBatch, F_LABEL_BITS
    from hdgnn_b200.model import truncated_normal_init
    Ne, Nc, B, variant = 200, 74, 8, 2
    cb = make_commits(B, Ne, Nc, seed=9)
    for extra in (0, F_LEGACY):
        out = []
        for flags in (0, F_LABEL_BITS):
            eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=flags | extra)
            db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev, bits=bool(flags))
            params = truncated_normal_init(variant, 3).cuda()
            m = torch.zeros_like(params); v = torch.zeros_like(params)
            step = torch.zeros(1, dtype=torch.int32, device="cuda"); loss3 = torch.zeros(3, device="cuda")
            probs = torch.zeros(B, 2, Nc * (Nc - 1), device="cuda")
            for _ in range(2):
                eng.train_step(db, params, m, v, step, loss3, probs=probs)
            p2, _, l2 = eng.forward(db, params, want_logits=False)
            torch.cuda.synchronize()
            out.append((params.cpu().numpy(), probs.cpu().numpy(), loss3.cpu().numpy(), p2.cpu().numpy(), l2.cpu().numpy(), eng.last_launch_count()))
            eng.close()
        for k in range(5):
            assert np.array_equal(out[0][k], out[1][k]), (extra, k)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, 8])        # byte grids (5 launches incl. pack_bits), label bitmaps (4 launches)
def test_train_step_is_cuda_graph_capturable_and_replayable(flags):
    """include/hdgnn.h promises asynchronous, capturable entry points: the whole training step (programmatic dependent
    launches included) is captured once and replayed; Adam's step count lives on the device, so replays advance it."""
    from hdgnn_b200.engine import Engine, DeviceBatch
    from hdgnn_b200.model import truncated_normal_init
    Ne, Nc, B, variant, steps = 64, 24, 6, 2, 4
    cb = make_commits(B, Ne, Nc, seed=21)
    res = []
    for mode in ("eager", "graph"):
        eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=flags)
        db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev, bits=bool(flags))
        params = truncated_normal_init(variant, 3).cuda()
        m = torch.zeros_like(params); v = torch.zeros_like(params)
        step = torch.zeros(1, dtype=torch.int32, device="cuda"); loss3 = torch.zeros(3, device="cuda")
        probs = torch.zeros(B, 2, Nc * (Nc - 1), device="cuda")
        if mode == "eager":
            for _ in range(steps):
                eng.train_step(db, params, m, v, step, loss3, probs=probs)
        else:
            eng.train_step(db, params, m, v, step, loss3, probs=probs)       # warm-up outside the capture (attributes, lazy init)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                eng.train_step(db, params, m, v, step, loss3, probs=probs)
            # the capture only recorded: one eager + (steps - 1) replays = `steps` steps
            for _ in range(steps - 1):
                g.replay()
        torch.cuda.synchronize()
        res.append((params.cpu().numpy(), m.cpu().numpy(), int(step.item()), loss3.cpu().numpy(), probs.cpu().numpy()))
        eng.close()
    assert res[0][2] == res[1][2] == steps
    for k in (0, 1, 3, 4):
        assert np.array_equal(res[0][k], res[1][k]), k
