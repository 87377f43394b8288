"""The scratch buffers a handle owns (hdgnn_workspace): each one exists only where a planned kernel uses it, the buffers the
debug dumps and tools read exist with the sizes they read, and asking for a buffer the handle does not have is an error."""
import ctypes as C

import pytest

from hdgnn_b200.synthetic import make_commits

pytestmark = pytest.mark.gpu

F_DEBUG, F_LEGACY, F_LABEL_BITS, F_DENSE = 2, 4, 8, 16
PATH_FLAGS = {"default": 0, "dense": F_DENSE, "legacy": F_LEGACY}
ENTITY_STATE = ("RS1", "CS1P", "GPE", "GE")


def _query(eng, name):
    """(return code, device pointer, bytes) of hdgnn_workspace"""
    from hdgnn_b200._lib import lib
    p, n = C.c_void_p(), C.c_size_t()
    rc = lib.hdgnn_workspace(eng._h, name.encode(), C.byref(p), C.byref(n))
    return rc, p.value, n.value


def _bytes(eng, name):
    """size of the buffer in bytes, None when the handle does not have it"""
    from hdgnn_b200._lib import OK
    rc, p, n = _query(eng, name)
    if rc != OK:
        return None
    assert p and n > 0, (name, p, n)
    return n


def _train_launches(eng, B):
    """launch count of one forward + backward on a batch of B commits"""
    import torch
    from hdgnn_b200.engine import DeviceBatch
    cb = make_commits(B, eng.Ne, eng.Nc, seed=5)
    db = DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev, bits=eng.host_bits)
    params = torch.zeros(eng.n_params, dtype=torch.float32, device=eng.tdev)
    eng.forward_backward(db, params)
    torch.cuda.synchronize()
    return eng.last_launch_count()


@pytest.mark.parametrize("flags", [0, F_LABEL_BITS])
def test_inline_entity_stage_keeps_entity_state_out_of_hbm(flags):
    """glide, variant 2: mid2 runs the entity pair layer inline and keeps S and GE in shared memory"""
    from hdgnn_b200.engine import Engine
    B, Ne, Nc = 100, 200, 74
    eng = Engine(Ne, Nc, variant=2, max_batch=B, flags=flags)
    assert {n: _bytes(eng, n) for n in ENTITY_STATE} == dict.fromkeys(ENTITY_STATE)
    assert _bytes(eng, "GPART") == 2 * B * eng.n_params * 4      # the cluster form parks rank 1's partials in the second half
    assert _train_launches(eng, 4) == (2 if flags else 3)        # [pack_bits], mid, reduce
    eng.close()


def test_dense_sweeps_keep_entity_state_in_hbm():
    from hdgnn_b200.engine import Engine
    B, Ne, Nc = 100, 200, 74
    eng = Engine(Ne, Nc, variant=2, max_batch=B, flags=F_DENSE)
    sizes = {n: _bytes(eng, n) for n in ENTITY_STATE}
    assert all(sizes.values()), sizes
    assert sizes["RS1"] == sizes["GE"] == B * Ne * 20 * 4
    assert _train_launches(eng, 4) == 5                           # pack_bits, ent_fwd, mid, ent_bwd, reduce
    eng.close()


@pytest.mark.parametrize("path", ["default", "dense", "legacy"])
@pytest.mark.parametrize("B,Ne,Nc,variant", [(2, 200, 74, 2), (2, 250, 150, 2), (2, 120, 170, 2), (2, 97, 74, 4), (3, 40, 20, 1)])
def test_debug_dump_targets_exist(B, Ne, Nc, variant, path):
    """HDGNN_F_DEBUG: every buffer test_gpu_parity reads, with the size it reads; CLK (tools/mid_phases.py) on the fused path"""
    from hdgnn_b200.engine import Engine
    if path == "dense" and variant != 2:
        pytest.skip("the dense-sweep flag only changes variant 2")
    eng = Engine(Ne, Nc, variant=variant, max_batch=B, flags=F_DEBUG | PATH_FLAGS[path])
    floats = {"NB": B * Nc * 4, "RS3": B * Nc * 20, "CS3F": B * Nc * 20, "PR": B * Nc * 20, "PC": B * Nc * 20,
              "DNB": B * Nc * 4}
    launches = _train_launches(eng, B)
    if variant in (2, 4):
        floats.update(S1=B * Ne * 20, X2=B * Ne, DX2=B * Ne, GE=B * Ne * 20)
        if path == "legacy" or launches >= 5:
            floats["RS1"] = B * Ne * 20
    got = {n: _bytes(eng, n) for n in floats}
    assert got == {n: 4 * f for n, f in floats.items()}
    if path != "legacy" and launches <= 5:
        assert _bytes(eng, "CLK") == B * 24 * 8
    eng.close()


def test_unfused_training_has_no_dlt():
    """variant 4 at Ne = 240, Nc = 104: the forward is fused, the training step runs on the multi-kernel path, and the dL/dlogit
    table that only the fused training kernel reads from HBM is not allocated"""
    from hdgnn_b200.engine import Engine
    eng = Engine(240, 104, variant=4, max_batch=2)
    assert _train_launches(eng, 2) > 5
    assert _bytes(eng, "DLT") is None
    eng.close()


def test_absent_and_unknown_names_are_errors():
    """a buffer this handle does not have (RS1 of variant 1, also after a step) and an unknown name: HDGNN_E_INVALID, each with
    its own message"""
    from hdgnn_b200._lib import lib, E_INVALID, HdgnnError
    from hdgnn_b200.engine import Engine
    eng = Engine(40, 20, variant=1, max_batch=3)
    _train_launches(eng, 3)
    rc, p, _ = _query(eng, "RS1")
    assert rc == E_INVALID and p is None
    assert b"not allocated" in lib.hdgnn_last_error(eng._h)
    rc, p, _ = _query(eng, "RS2")
    assert rc == E_INVALID and p is None
    assert b"no workspace buffer named RS2" in lib.hdgnn_last_error(eng._h)
    with pytest.raises(HdgnnError):
        eng.workspace("RS1", (3, 40, 20))
    assert _bytes(eng, "CEP") is not None
    eng.close()
