"""graph2graph -- host-side mirror of the reference's model class (model_2.py:15-544 and the
model_1/3/4 ablations) over the B200 engine.

Same constructor keywords, same train(args)/test(args)/save/load surface, same output files and
log lines; the numeric work of every `sess.run` (model_2.py:369-383, 486-502) is one call into
libhdgnn (include/hdgnn.h).  Commits are sharded across ranks when torch.distributed is
initialised; the only collective is one all-reduce of the flat gradient per step.
"""
from __future__ import annotations

import os
import time
from typing import Optional

import numpy as np
import torch

from .engine import Engine, DeviceBatch, param_count, param_offsets, PARAM_NAMES, F_LABEL_BITS, F_DENSE_SWEEP, pack_label_bits
from .synthetic import CommitBatch

H = 20

_SHAPES = {
    "ent_w1": (4, H), "ent_b1": (H,), "ent_w5": (H, H), "ent_b5": (H,), "nod_w1": (H + 1, H), "nod_b1": (H,),
    "nod_w2": (H, 1), "nod_b2": (1,), "edg_w11": (1, H), "edg_w12": (2, H), "edg_b1": (H,), "edg_w2": (H, H),
    "edg_b2": (H,), "eup_w1": (H + 2, H), "eup_b1": (H,), "eup_w2": (H, 2), "eup_b2": (2,),
    "hnk_w1": (10, H), "hnk_b1": (H,), "hnk_w2": (H, H), "hnk_b2": (H,), "scr_w1": (H + 2, H), "scr_b1": (H,),
    "scr_w2": (H, 2), "scr_b2": (2,), "theta1": (2,), "theta2": (2,),
}
# tf scope/name of every block (model_2.py:167-201, 257-264, 311-319, 329-330; model_4.py:219-229, 292-297)
TF_NAMES = {
    "ent_w1": "phi_E_O1/r1_w1o", "ent_b1": "phi_E_O1/r1_b1o", "ent_w5": "phi_E_O1/r1_w5o", "ent_b5": "phi_E_O1/r1_b5o",
    "nod_w1": "phi_U_O1/o1_w1o", "nod_b1": "phi_U_O1/o1_b1o", "nod_w2": "phi_U_O1/o1_w2o", "nod_b2": "phi_U_O1/o1_b2o",
    "edg_w11": "phi_E_R1/r1_w1r1", "edg_w12": "phi_E_R1/r1_w1r2", "edg_b1": "phi_E_R1/r1_b1r",
    "edg_w2": "phi_E_R1/r1_w2r", "edg_b2": "phi_E_R1/r1_b2r", "eup_w1": "phi_U_R1/o1_w1r", "eup_b1": "phi_U_R1/o1_b1r",
    "eup_w2": "phi_U_R1/o1_w2r", "eup_b2": "phi_U_R1/o1_b2r",
    "hnk_w1": "mlp_hunk_B2/w1", "hnk_b1": "mlp_hunk_B2/b1", "hnk_w2": "mlp_hunk_B2/r1_w2r", "hnk_b2": "mlp_hunk_B2/b2",
    "scr_w1": "phi_U_R1/C_edge_w1", "scr_b1": "phi_U_R1/C_edge_b1", "scr_w2": "phi_U_R1/o1_w2r", "scr_b2": "phi_U_R1/o1_b2r",
    "theta1": "map_conv/map_theta1", "theta2": "map_conv/map_theta2",
}


def truncated_normal_init(variant: int, seed: Optional[int] = None) -> torch.Tensor:
    """tf.truncated_normal(stddev=0.1) weights, tf.zeros biases (model_2.py:167-201); values beyond
    two standard deviations are re-drawn.  The reference is unseeded; `seed` makes runs repeatable."""
    g = torch.Generator()
    if seed is None:
        g.seed()
    else:
        g.manual_seed(seed)
    parts = []
    for name in PARAM_NAMES[variant]:
        n = int(np.prod(_SHAPES[name]))
        if "_b" in name:
            parts.append(torch.zeros(n))
            continue
        v = torch.randn(n, generator=g)
        bad = v.abs() > 2
        while bad.any():
            v[bad] = torch.randn(int(bad.sum()), generator=g)
            bad = v.abs() > 2
        parts.append(0.1 * v)
    return torch.cat(parts)


class HostBatch:
    """Pinned host copy of a compact commit batch (the wire format into the hot path).  bits=True: the two label
    grids travel as bitmaps (HDGNN_F_LABEL_BITS, 1/8 of the bytes); Y is kept as bytes too for the evaluation kernel.
    With bitmaps the five arrays sit back to back in ONE pinned block, every array starting at the next multiple of 16 bytes in
    the order adj, Y, x, hmap, L -- the layout the library's staging slot has, so a step's inputs travel in a single DMA
    (include/hdgnn.h, the *_host entry points)."""

    def __init__(self, cb: CommitBatch, bits: bool = False):
        self.bits = bits
        self.Y = self._pin(torch.as_tensor(np.ascontiguousarray(cb.Y, dtype=np.uint8)))
        if bits:
            self._fill(pack_label_bits(cb.adj).view(np.int32), pack_label_bits(cb.Y).view(np.int32), cb.x, cb.hmap, cb.L)
        else:
            mk = lambda a, dt: self._pin(torch.as_tensor(np.ascontiguousarray(a, dtype=dt)))
            self.adj, self.Yw = mk(cb.adj, np.uint8), self.Y
            self.x = mk(cb.x, np.float32)
            self.hmap, self.L = mk(cb.hmap, np.int32), mk(cb.L, np.int32)
        self.B = self.adj.shape[0]

    @staticmethod
    def _pin(t):
        return t.pin_memory() if torch.cuda.is_available() else t

    def _fill(self, adj, Yw, x, hmap, L):
        """adj, Yw int32 bitmaps; x float32; hmap, L int32 (numpy or torch): copies them into one pinned block."""
        parts = [torch.as_tensor(np.ascontiguousarray(a)) if not torch.is_tensor(a) else a.contiguous() for a in (adj, Yw, x, hmap, L)]
        parts = [p.to(dt) for p, dt in zip(parts, (torch.int32, torch.int32, torch.float32, torch.int32, torch.int32))]
        offs, o = [], 0
        for p in parts:
            offs.append(o)
            o += (p.numel() * p.element_size() + 15) & ~15
        block = self._pin(torch.zeros(max(o, 16), dtype=torch.uint8))
        views = []
        for p, off in zip(parts, offs):
            n = p.numel() * p.element_size()
            v = block[off:off + n].view(p.dtype).view(p.shape)
            v.copy_(p)
            views.append(v)
        self._block = block
        self.adj, self.Yw, self.x, self.hmap, self.L = views

    def clone(self) -> "HostBatch":
        """Same batch in freshly pinned buffers."""
        c = object.__new__(HostBatch)
        c.bits, c.B = self.bits, self.B
        c.Y = self._pin(self.Y.clone())
        if self.bits:
            c._fill(self.adj, self.Yw, self.x, self.hmap, self.L)
        else:
            for k in ("adj", "x", "hmap", "L"):
                setattr(c, k, self._pin(getattr(self, k).clone()))
            c.Yw = c.Y
        return c

    def nbytes(self):
        """bytes copied host -> device per step"""
        return sum(t.numel() * t.element_size() for t in self.tensors())

    def tensors(self):
        return self.adj, self.x, self.hmap, self.L, self.Yw


class graph2graph(object):
    def __init__(self, sess=None, Ds=1, Ne=200, Nc=74, Ner=None, Ncr=None, Dr=2, De_e=20, De_er=20, Mini_batch=50,
                 checkpoint_dir="./checkpoint40/", epoch=50, Ds_inter=1, Dr_inter=2, Step=2, Repo="glide",
                 variant=2, device: Optional[int] = None, seed: Optional[int] = None, max_batch: Optional[int] = None,
                 collective: str = "auto", entity_sweep: str = "auto"):
        # `sess` is accepted and ignored: there is no TF session (main.py:54-56).
        Ner = Ne * (Ne - 1) if Ner is None else Ner
        Ncr = Nc * (Nc - 1) if Ncr is None else Ncr
        if Ner != Ne * (Ne - 1) or Ncr != Nc * (Nc - 1):
            raise ValueError(f"Ner/Ncr must be Ne(Ne-1)/Nc(Nc-1) (utils2.py:69-83): got Ne={Ne} Ner={Ner} Nc={Nc} Ncr={Ncr}")
        if (Ds, Ds_inter, Dr, Dr_inter, De_e, De_er) != (1, 1, 2, 2, 20, 20):
            raise ValueError("the sm_100a kernels are specialised to the reference's dimensions "
                             "Ds=Ds_inter=1, Dr=Dr_inter=2, De_e=De_er=20 (main.py:26-32; model_2.py:200-203 "
                             "silently requires Ds==Ds_inter, Dr==Dr_inter)")
        if variant not in (1, 2, 3, 4):
            raise ValueError("variant must be 1 (model_1), 2 (model_2), 3 (model_3) or 4 (model_4)")
        self.sess = sess
        self.Ds, self.Ne, self.Nc, self.Ner, self.Ncr, self.Dr = Ds, Ne, Nc, Ner, Ncr, Dr
        self.Ds_inter, self.Dr_inter, self.De_e, self.De_er = Ds_inter, Dr_inter, De_e, De_er
        self.mini_batch_num = Mini_batch
        self.epoch = epoch
        self.checkpoint_dir = checkpoint_dir
        self.Step, self.Repo = Step, Repo
        self.variant = variant
        self.seed = seed
        self.world = torch.distributed.get_world_size() if torch.distributed.is_initialized() else 1
        self.rank = torch.distributed.get_rank() if torch.distributed.is_initialized() else 0
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0")) if self.world > 1 else 0
        self.device = device
        self.max_batch = max_batch or Mini_batch
        if collective not in ("auto", "peer", "nccl"):
            raise ValueError("collective must be 'auto', 'peer' (all-reduce fused into the last kernel over NVLink peer "
                             "memory) or 'nccl' (torch.distributed.all_reduce between backward and Adam)")
        self.collective = collective
        if entity_sweep not in ("auto", "inline", "dense"):
            raise ValueError("entity_sweep must be 'auto', 'inline' (sorted prefix sums / class tables inside the per-commit kernel) "
                             "or 'dense' (the Ne x Ne sweep kernels, HDGNN_F_DENSE_SWEEP)")
        self.entity_sweep = entity_sweep
        self._dense = entity_sweep == "dense"
        self._saved = {}                 # checkpoint dir -> names written by THIS object (the Saver's max_to_keep list)
        self.build_model()

    # ------------------------------------------------------------------------------------------
    def build_model(self):
        torch.cuda.set_device(self.device)
        # label grids as bitmaps on the wire (1/8 of the H2D bytes, no packing kernel)
        self.engine = Engine(self.Ne, self.Nc, variant=self.variant, max_batch=self.max_batch, device=self.device,
                             flags=F_LABEL_BITS | (F_DENSE_SWEEP if self._dense else 0))
        self.host_bits = self.engine.host_bits
        self.n_params = param_count(self.variant)
        self.offsets = param_offsets(self.variant)
        dev = self.engine.tdev
        self.params = torch.empty(self.n_params, dtype=torch.float32, device=dev)
        self.m = torch.zeros_like(self.params)
        self.v = torch.zeros_like(self.params)
        self.grads = torch.zeros_like(self.params)
        self.step_counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self.reg = torch.zeros(2, dtype=torch.float32, device=dev)
        self.loss_d = torch.zeros(1, dtype=torch.float32, device=dev)
        self.loss3 = torch.zeros(3, dtype=torch.float32).pin_memory()
        # gradient exchange of the sharded step: peer memory (one fused kernel) when every rank can map its peers
        self.peer = self.world > 1 and self.collective != "nccl" and self.engine.peer_attach(self.collective)
        self.initialize()

    def initialize(self, flat: Optional[torch.Tensor] = None):
        """tf.global_variables_initializer (model_2.py:340-341): fresh weights, Adam slots zeroed."""
        if flat is None:
            flat = truncated_normal_init(self.variant, self.seed)
            if self.world > 1:      # every rank must start from the same weights
                t = flat.to(self.engine.tdev)
                torch.distributed.broadcast(t, 0)
                flat = t
        assert flat.numel() == self.n_params
        self.params.copy_(flat.to(torch.float32))
        self.m.zero_(); self.v.zero_(); self.step_counter.zero_()

    def host_batch(self, cb: CommitBatch) -> HostBatch:
        """Pinned host batch in the wire format this model's engine takes."""
        return HostBatch(cb, bits=self.host_bits)

    def named_params(self, flat=None):
        out = {}
        flat = self.params.detach().cpu() if flat is None else torch.as_tensor(flat)
        for name in PARAM_NAMES[self.variant]:
            o = self.offsets[name]
            out[name] = flat[o:o + int(np.prod(_SHAPES[name]))].reshape(_SHAPES[name]).clone()
        return out

    # ------------------------------------------------------------------------------------------
    # one `sess.run([... trainer])` (model_2.py:369-383)
    def train_step(self, hb: HostBatch, want_probs: bool = False, probs_out: Optional[torch.Tensor] = None):
        """hb: this rank's shard of the global batch (pinned host tensors).  Returns the pinned
        3-vector {CE (this rank's share of the global mean), loss_map, loss_para}; valid after a
        stream synchronize.  probs_out: pinned host OR device tensor (>= (B,2,Ncr)) that receives the probabilities."""
        eng = self.engine
        if self.world == 1:
            eng.train_step_host(*hb.tensors(), self.params, self.m, self.v, self.step_counter, self.loss3,
                                probs=probs_out if want_probs else None)
            return self.loss3
        if self.peer:                                   # loss3[0] is already the global mean CE
            eng.train_step_peer_host(*hb.tensors(), self.params, self.m, self.v, self.step_counter, self.loss3,
                                     probs=probs_out if want_probs else None)
            return self.loss3
        direct = want_probs and probs_out is not None and probs_out.is_cuda
        if want_probs and not direct and (not hasattr(self, "_probs_d") or self._probs_d.shape[0] < hb.B):
            self._probs_d = torch.zeros(hb.B, 2, self.Ncr, dtype=torch.float32, device=eng.tdev)
        pd = (probs_out if direct else self._probs_d) if want_probs else None
        eng.forward_backward_host(*hb.tensors(), self.params, self.grads, hb.B * self.world, loss=self.loss_d, probs=pd)
        torch.distributed.all_reduce(self.grads)        # the single collective of the step
        eng.adam_step(self.params, self.grads, self.m, self.v, self.step_counter, reg_losses=self.reg)
        self.loss3[0:1].copy_(self.loss_d, non_blocking=True)
        self.loss3[1:3].copy_(self.reg, non_blocking=True)
        if want_probs and probs_out is not None and not direct:
            probs_out.copy_(self._probs_d[:hb.B], non_blocking=True)
        return self.loss3

    # one `sess.run([loss, loss_map, probs])` (model_2.py:486-502)
    def infer(self, hb: HostBatch, probs_out: torch.Tensor, loss_out: Optional[torch.Tensor] = None):
        self.engine.infer_host(*hb.tensors(), self.params, probs_out, loss_out)

    # ------------------------------------------------------------------------------------------
    # data
    def _load(self, root="."):
        from .utils2 import read_compact, split_half
        cb = read_compact(self.Repo, self.Step, self.Ne, self.Nc, root=root, device=self.engine.tdev)
        return split_half(cb)

    def _batch(self, part: CommitBatch, maps: CommitBatch, j: int, quirk_q2: bool) -> CommitBatch:
        """Batch j of `part`; with quirk Q2 (model_2.py:376-381, 495-500) the entity->hunk maps are always
        those of the first Mini_batch commits of the whole data set."""
        mb = self.mini_batch_num
        lo = j * mb
        src = maps.slice(0, mb) if quirk_q2 else part.slice(lo, lo + mb)
        b = CommitBatch(part.adj[lo:lo + mb], part.x[lo:lo + mb], src.hmap, src.L, part.Y[lo:lo + mb])
        if self.world > 1:                       # this rank's contiguous shard of the global batch
            per = mb // self.world
            b = b.slice(self.rank * per, (self.rank + 1) * per)
        return b

    def _choose_entity_sweep(self, cb: CommitBatch):
        """entity_sweep='auto': the inline entity stage costs O(edges) when the node attribute has more than 16 distinct
        values per commit (class tables otherwise), the dense sweeps O(Ne^2): measured break-even near 15-20 % edge density
        (tools/step_probe.py).  Decided from the data set, identically on every rank; rebuilds the engine if it changes."""
        if self.entity_sweep != "auto" or self.variant != 2 or cb.B == 0:
            return
        n = min(cb.B, 64)
        distinct = max(len(np.unique(cb.x[b])) for b in range(n))
        density = float(np.asarray(cb.adj[:n], dtype=np.float32).mean())
        dense = distinct > 16 and density > 0.15
        if dense != self._dense:
            self._dense = dense
            params = self.params.clone()
            self.engine.close()
            self.build_model()
            self.params.copy_(params)

    def _model_dir(self):
        return "%s" % (self.Repo + '/model_%d/' % self.variant + str(self.Step))

    # ------------------------------------------------------------------------------------------
    def train(self, args=None, data=None, root=".", quirk_q2=True, log=print, save_checkpoints=True):
        """model_2.py:335-424.  `args` needs .Repo and .checkpoint_dir (main.py's namespace).
        The loop body is one asynchronous library call per batch: the batches are pinned (and bit-packed) once, the losses of
        an epoch land in a pinned ring, top_ACC (EvaluationFuncs.py:27-37) is counted inside the relation-head phase of the
        step (hdgnn_set_hits_accumulator).  The host never waits for the epoch it has just enqueued: at the end of epoch i
        the parameters / Adam state / hit count are copied to pinned memory asynchronously and an event is recorded; the log
        line, the result file and the checkpoint of epoch i are written while epoch i+1 runs (same order, same content)."""
        from .engine import eval_counts
        repo = getattr(args, "Repo", self.Repo)
        ckpt = getattr(args, "checkpoint_dir", self.checkpoint_dir)
        self.initialize()                                           # always from scratch (model_2.py:340-341)
        train, _ = data if data is not None else self._load(root)
        self._choose_entity_sweep(train)
        mb = self.mini_batch_num
        if self.world > 1 and mb % self.world:
            raise ValueError("Mini_batch must be divisible by the number of ranks")
        nb = int(train.B / mb)                                      # remainder batch dropped (model_2.py:364)
        per = mb // self.world
        dev = self.engine.tdev
        E, P = self.epoch, self.n_params
        hits_dev = torch.zeros(max(E, 1), dtype=torch.int64, device=dev)          # one counter per epoch: no memset in the loop
        in_kernel_hits = self.engine.set_hits_accumulator(hits_dev[0:1])          # False on the multi-kernel path (very large grids)
        probs_d = None if in_kernel_hits else torch.zeros(per, 2, self.Ncr, dtype=torch.float32, device=dev)
        ring = torch.zeros(2, max(nb, 1), 3, dtype=torch.float32).pin_memory()    # losses, by epoch parity
        snap = torch.zeros(2, 3 * P + 1, dtype=torch.float32).pin_memory()        # params | m | v | step count at the end of an epoch
        hits_h = torch.zeros(2, dtype=torch.int64).pin_memory()
        done = [torch.cuda.Event(), torch.cuda.Event()]
        side = torch.cuda.Stream(device=dev) if self.world > 1 else None
        keep3 = self.loss3
        history = []
        # the data set is static across epochs: pin (and bit-pack) every batch once
        batches = [self.host_batch(self._batch(train, train, j, quirk_q2)) for j in range(nb)]
        y_dev = None if in_kernel_hits else [hb.Y.to(dev) for hb in batches]
        o2 = self.offsets["theta2"]
        if self.world > 1:
            torch.distributed.barrier()          # data preparation can skew the ranks by seconds: line up before the first exchange

        def finish(i):
            """Log line, result file and checkpoint of epoch i (its event has been recorded)."""
            s = i & 1
            done[s].synchronize()
            ce_steps = ring[s, :nb, 0].double()
            nhits = int(hits_h[s].item())
            if self.world > 1:                                      # on a side stream: the training stream keeps running
                with torch.cuda.stream(side):
                    t = torch.cat([ce_steps if not self.peer else torch.zeros(0, dtype=torch.float64),
                                   torch.tensor([float(nhits)], dtype=torch.float64)]).to(dev)
                    torch.distributed.all_reduce(t)
                    t = t.cpu()
                if not self.peer:                                   # CE partials add up to the global mean
                    ce_steps = t[:nb]
                nhits = int(round(float(t[-1])))
            tr_loss_Hedge = float(ce_steps.sum())
            tr_loss_map = float(ring[s, :nb, 1].double().sum())
            acc_top = float(nhits / (nb * mb * self.Ncr)) if nb else float("nan")
            flat = snap[s, :P]
            theta = flat[o2:o2 + 2].numpy().copy()
            resultString = "Epoch " + str(i + 1) + \
                           " acc: " + str(acc_top)[0:6] + \
                           " Hedge loss: " + str(tr_loss_Hedge / nb)[0:6] + \
                           " map MSE: " + str(tr_loss_map / nb)[0:6] + \
                           " theta: " + str(theta[0]) + ' ' + str(theta[1]) + '\n'
            history.append(dict(epoch=i + 1, acc=acc_top, hedge_loss=tr_loss_Hedge / nb, map_loss=tr_loss_map / nb))
            if self.rank == 0 and save_checkpoints:
                filepath = r'outputSelf/{}/model_{}/{}/result_{}.npy'.format(repo, self.variant, self.Step, self.Step)
                filepath = os.path.join(root, filepath)
                os.makedirs(os.path.dirname(filepath), exist_ok=True)
                with open(filepath, "a", encoding='utf-8') as f:
                    f.write(resultString)
            if self.rank == 0:
                log(resultString)
            if self.rank == 0 and save_checkpoints:                 # counter = i + 2: the reference increments before saving
                self.save(os.path.join(root, ckpt) if not os.path.isabs(ckpt) else ckpt, i + 2,
                          snapshot=dict(params=flat.clone(), m=snap[s, P:2 * P].clone(), v=snap[s, 2 * P:3 * P].clone(),
                                        t=np.array([int(round(float(snap[s, 3 * P])))], dtype=np.int32)))

        start_time1 = time.time()
        try:
            for i in range(E):
                s = i & 1
                if in_kernel_hits:
                    self.engine.set_hits_accumulator(hits_dev[i:i + 1])
                for j in range(nb):
                    hb = batches[j]
                    self.loss3 = ring[s, j]
                    if in_kernel_hits:
                        self.train_step(hb)
                    else:
                        self.train_step(hb, want_probs=True, probs_out=probs_d)
                        counts, _ = eval_counts(probs_d[:hb.B], y_dev[j])
                        hits_dev[i:i + 1] += counts[:, 0].sum()
                snap[s, :P].copy_(self.params, non_blocking=True)
                if save_checkpoints:
                    snap[s, P:2 * P].copy_(self.m, non_blocking=True)
                    snap[s, 2 * P:3 * P].copy_(self.v, non_blocking=True)
                    snap[s, 3 * P:].copy_(self.step_counter.float(), non_blocking=True)
                hits_h[s:s + 1].copy_(hits_dev[i:i + 1], non_blocking=True)
                done[s].record()
                if i >= 1:
                    finish(i - 1)                                   # while epoch i runs
                if self.peer and (i & 31) == 31:
                    self.engine.peer_status()    # a timed-out exchange raises here instead of training on with diverged replicas
            if E:
                finish(E - 1)
            if self.peer:
                self.engine.peer_status()
        finally:
            self.loss3 = keep3
            self.engine.set_hits_accumulator(None)
        end_time1 = time.time()
        self.last_train_seconds = end_time1 - start_time1          # the epoch loop alone, as the reference times it (model_2.py:358,423)
        if self.rank == 0:
            log('test time:' + str(end_time1 - start_time1))       # sic (model_2.py:424)
        return history

    def test(self, args=None, data=None, root=".", quirk_q2=True, quirks=True, log=print):
        """model_2.py:453-544: inference over the test half, writes C_edge_t{Ne}.npy / C_edge_y{Ne}.npy and
        prints the metric lines.  The metrics come from integer counters computed on the device
        (hdgnn_eval_counts); the probabilities are copied back once, for the output file only."""
        from .EvaluationFuncs import metrics_from_counts, auc_from_counts
        from .engine import eval_counts
        from .utils2 import edge_onehot
        repo = getattr(args, "Repo", self.Repo)
        train, test = data if data is not None else self._load(root)
        self.initialize()
        ckroot = self.checkpoint_dir if os.path.isabs(self.checkpoint_dir) else os.path.join(root, self.checkpoint_dir)
        checkpoint_dir = os.path.join(ckroot, self.Repo)            # model_2.py:464 (path quirk Q8)
        if self.load(checkpoint_dir) or self.load(ckroot, note=" [*] (found under the directory save() writes to)"):
            log(" [*] Load SUCCESS")
        else:
            log(" [!] Load failed...")
        mb = self.mini_batch_num
        nb = int(test.B / mb)
        n = nb * mb
        dev = self.engine.tdev
        probs_d = torch.zeros(max(n, 1), 2, self.Ncr, dtype=torch.float32, device=dev)
        counts_d = torch.zeros(max(n, 1), 8, dtype=torch.int64, device=dev)
        auc_d = torch.zeros(max(n, 1), 2, dtype=torch.int64, device=dev)
        loss_h = torch.zeros(max(nb, 1)).pin_memory()
        start_time = time.time()
        alive = []       # the library DMAs from these pinned buffers asynchronously: keep them until the final synchronize
        # top_ACC / prec / recall / f1 counters come out of the relation head itself (hdgnn_set_eval_counters: no second kernel,
        # no label bytes on the device); only the batches whose AUC is wanted run hdgnn_eval_counts as well
        in_kernel = self.engine.set_eval_counters(counts_d[0:mb]) if nb else False
        for j in range(nb):
            saved = (self.world, self.rank)
            self.world, self.rank = 1, 0                            # inference is not sharded
            hb = self.host_batch(self._batch(test, train, j, quirk_q2))
            self.world, self.rank = saved
            alive.append(hb)
            pj = probs_d[j * mb:(j + 1) * mb]
            if in_kernel:
                self.engine.set_eval_counters(counts_d[j * mb:(j + 1) * mb])
            self.infer(hb, pj, loss_h[j:j + 1])
            # the reference's AUC keeps only the last commit of the whole test set (quirk Q7)
            first = (mb - 1 if j == nb - 1 else mb) if quirks else 0
            if not in_kernel or first < mb:
                c, a = eval_counts(pj, hb.Y.to(dev, non_blocking=True), auc=True, auc_first=first)
                if not in_kernel:
                    counts_d[j * mb:(j + 1) * mb] = c
                auc_d[j * mb:(j + 1) * mb] = a
        if in_kernel:
            self.engine.set_eval_counters(None)
        torch.cuda.current_stream().synchronize()
        alive.clear()
        end_time = time.time()
        te_loss_Hedge = float(loss_h[:nb].sum())
        C_edge_t1 = probs_d[:n].cpu().numpy().reshape(n, self.Dr, self.Ncr) if nb else np.zeros((0, 2, self.Ncr), np.float32)
        out = {}
        if self.rank == 0:
            C_edge_test = edge_onehot(test.Y[:n])
            step_dir = os.path.join(root, 'outputSelf/' + repo + '/model_%d/' % self.variant + str(self.Step) + '/')
            os.makedirs(step_dir, exist_ok=True)
            np.save(step_dir + 'C_edge_t' + str(self.Ne) + '.npy', C_edge_t1)
            np.save(step_dir + 'C_edge_y' + str(self.Ne) + '.npy', C_edge_test)
            counts, auc = counts_d[:n].cpu().numpy(), auc_d[:n].cpu().numpy()
            m = metrics_from_counts(counts, quirks) if nb else dict(hits=0, prec=float("nan"), recall=float("nan"), f1=float("nan"))
            out = dict(topol_acc=m["hits"] / max(n * self.Ncr, 1), prec=m["prec"], recall=m["recall"], f1=m["f1"],
                       hedge_loss=te_loss_Hedge / max(nb, 1), counts=counts)
            try:
                out["auc"] = auc_from_counts(counts, auc, self.Ncr, quirks) if nb else float("nan")
            except ZeroDivisionError:
                out["auc"] = float("nan")
            log('topol_acc: ' + str(out["topol_acc"]))
            log('prec: ' + str(out["prec"]))
            log('recall: ' + str(out["recall"]))
            log('F1-score: ' + str(out["f1"]))
            log('AUC-score: ' + str(out["auc"]))
            log('test time:' + str(end_time - start_time))
        return out, C_edge_t1

    def untangle(self, args=None, data=None, root=".", quirk_q2=True, log=print, grouping="components", threshold=0.5,
                 sweep=None):
        """The untangling answer over the test half, with the checkpoint, batches and entity->hunk maps of test(): the predicted
        relations of every commit as a label bitmap (hdgnn_set_predictions; by default no probabilities are written) and the
        hunk groups they give (hdgnn_hunk_groups), beside the groups of the labels.  Writes C_group_t{Ne}.npy (predicted groups) and
        C_group_y{Ne}.npy (labelled groups), (n_test, Nc) int32, each hunk labelled with the smallest hunk index of its group, over
        all Nc hunks, and logs the number of commits whose predicted partition of all Nc hunks equals the labelled one
        (exact_partitions).  The group-level scores (hdgnn_partition_counts -> EvaluationFuncs.partition_metrics_from_counts:
        pair precision / recall / F1, Rand and adjusted Rand index, purity, groups per commit; out["partition_counts"] and
        out["partition"], one log line each before exact_partitions) count only each commit's real hunks 0 .. nh-1, the hunk
        count the loader read from the commit's hunk map (test.nh); padding hunks, singletons on both sides, would inflate every
        agreement measure.  A loader without hunk counts (test.nh None) scores all Nc hunks.
        grouping="components" forms the predicted groups as above.  grouping="average" forms them by average-linkage clustering
        of the relation probabilities (hdgnn_hunk_clusters) over the same real hunks: two groups merge only while the mean of
        max(p1(s,t), p1(t,s)) over their hunk pairs is > threshold, so one confident cross pair cannot join two groups and a few
        missing pairs cannot split one.  Each batch's probabilities go to a device buffer (never to the host); pred_bits keep
        their meaning, and one log line names the grouping before the partition_* lines.
        sweep (grouping="average" only): a sequence of further thresholds to score.  Each batch then runs hunk_linkage once and
        linkage_cut at [threshold, *sweep]; the groups at `threshold` are those of hunk_clusters, so everything above is
        unchanged.  Every sweep threshold is scored like the groups (out["sweep"]: threshold -> partition metrics, in the order
        given), and so is the cut at the labelled number of groups of each commit's real hunks (out["sweep_labelled_k"]: the
        score with the number of concerns known).  out["linkage"] = (merges, heights, nmerges) of every commit, also written as
        C_linkage{Ne}.npz; one log line per sweep threshold and one for the labelled-k cut come before the grouping line."""
        from .EvaluationFuncs import partition_metrics_from_counts
        from .engine import bit_words, hunk_clusters, hunk_groups, hunk_linkage, linkage_cut, partition_counts
        if grouping not in ("components", "average"):
            raise ValueError(f"grouping must be 'components' or 'average', got {grouping!r}")
        if sweep is not None:
            if grouping != "average":
                raise ValueError("sweep needs grouping='average'")
            sweep = [float(t) for t in sweep]
        repo = getattr(args, "Repo", self.Repo)
        train, test = data if data is not None else self._load(root)
        self.initialize()
        ckroot = self.checkpoint_dir if os.path.isabs(self.checkpoint_dir) else os.path.join(root, self.checkpoint_dir)
        if self.load(os.path.join(ckroot, self.Repo)) or self.load(ckroot, note=" [*] (found under the directory save() writes to)"):
            log(" [*] Load SUCCESS")
        else:
            log(" [!] Load failed...")
        mb = self.mini_batch_num
        nb = int(test.B / mb)
        n = nb * mb
        dev = self.engine.tdev
        pred = torch.zeros(max(n, 1), self.Nc, bit_words(self.Nc), dtype=torch.int32, device=dev)
        groups = torch.zeros(max(n, 1), self.Nc, dtype=torch.int32, device=dev)
        label_groups = torch.zeros_like(groups)
        pcounts = torch.zeros(max(n, 1), 8, dtype=torch.int64, device=dev)
        # the hunk counts of the commits whose labels Y are scored (never those of the Q2-substituted maps)
        nh = None if test.nh is None or not nb else torch.as_tensor(np.ascontiguousarray(test.nh[:n], dtype=np.int32)).to(dev)
        average = grouping == "average"
        probs = torch.empty(mb, 2, self.Ncr, dtype=torch.float32, device=dev) if average and nb else None
        if sweep is not None:
            link = (torch.full((max(n, 1), self.Nc - 1, 2), -1, dtype=torch.int32, device=dev),
                    torch.full((max(n, 1), self.Nc - 1), float("nan"), dtype=torch.float32, device=dev),
                    torch.zeros(max(n, 1), dtype=torch.int32, device=dev))
            scounts = torch.zeros(len(sweep) + 1, max(n, 1), 8, dtype=torch.int64, device=dev)   # the sweep, then labelled k
        start_time = time.time()
        alive = []       # the library DMAs from these pinned buffers asynchronously: keep them until the final synchronize
        try:
            for j in range(nb):
                saved = (self.world, self.rank)
                self.world, self.rank = 1, 0                        # inference is not sharded
                hb = self.host_batch(self._batch(test, train, j, quirk_q2))
                self.world, self.rank = saved
                alive.append(hb)
                rows = slice(j * mb, (j + 1) * mb)
                self.engine.set_predictions(pred[rows])
                self.engine.infer_host(*hb.tensors(), self.params, probs, None)
                nh_j = None if nh is None else nh[rows]
                if sweep is not None:
                    rec = hunk_linkage(probs, nh_j)
                    for dst, src in zip(link, rec):
                        dst[rows] = src
                    cuts = linkage_cut(*rec, nh_j, thresholds=[threshold, *sweep])[0]
                    groups[rows] = cuts[0]
                elif average:
                    groups[rows] = hunk_clusters(probs, nh_j, threshold)[0]
                else:
                    groups[rows] = hunk_groups(pred[rows])[0]
                label_groups[rows] = hunk_groups(hb.Yw.to(dev, non_blocking=True))[0]
                pcounts[rows] = partition_counts(groups[rows], label_groups[rows], nh_j)
                if sweep is not None:
                    for k in range(len(sweep)):
                        scounts[k, rows] = partition_counts(cuts[k + 1], label_groups[rows], nh_j)
                    # the labelled groups of the real hunks: column 5 of the counts just computed
                    at_k = linkage_cut(*rec, nh_j, target=pcounts[rows, 5].to(torch.int32))[0][0]
                    scounts[-1, rows] = partition_counts(at_k, label_groups[rows], nh_j)
        finally:
            self.engine.set_predictions(None)
        exact = int((groups[:n] == label_groups[:n]).all(1).sum()) if nb else 0      # synchronises
        alive.clear()
        end_time = time.time()
        out = dict(pred_bits=pred[:n].cpu().numpy(), groups=groups[:n].cpu().numpy(),
                   label_groups=label_groups[:n].cpu().numpy(), exact_partitions=exact,
                   partition_counts=pcounts[:n].cpu().numpy())
        out["partition"] = partition_metrics_from_counts(out["partition_counts"])
        if sweep is not None:
            sc = scounts[:, :n].cpu().numpy()
            out["sweep"] = {t: partition_metrics_from_counts(sc[k]) for k, t in enumerate(sweep)}
            out["sweep_labelled_k"] = partition_metrics_from_counts(sc[-1])
            out["linkage"] = tuple(x[:n].cpu().numpy() for x in link)
        if self.rank == 0:
            step_dir = os.path.join(root, 'outputSelf/' + repo + '/model_%d/' % self.variant + str(self.Step) + '/')
            os.makedirs(step_dir, exist_ok=True)
            np.save(step_dir + 'C_group_t' + str(self.Ne) + '.npy', out["groups"])
            np.save(step_dir + 'C_group_y' + str(self.Ne) + '.npy', out["label_groups"])
            if sweep is not None:
                np.savez(step_dir + 'C_linkage' + str(self.Ne) + '.npz', **dict(zip(("merges", "heights", "nmerges"), out["linkage"])))
                for t, v in out["sweep"].items():
                    log('sweep threshold ' + str(t) + ': ' + str(v))
                log('sweep labelled groups: ' + str(out["sweep_labelled_k"]))
            if average:
                log('grouping: average linkage, threshold ' + str(threshold))
            for k, v in out["partition"].items():
                log('partition_' + k + ': ' + str(v))
            log('exact_partitions: ' + str(exact) + ' / ' + str(n))
            log('test time:' + str(end_time - start_time))
        return out

    # ------------------------------------------------------------------------------------------
    # checkpoints: same directory layout and naming as tf.train.Saver (model_2.py:427-451), as .npz
    def save(self, checkpoint_dir, step, snapshot=None):
        """snapshot: host copies dict(params, m, v, t) taken at the end of the epoch (train() passes them so that the file
        is written while the next epoch runs); None reads the device state now."""
        model_name = "g2g.model"
        checkpoint_dir = os.path.join(checkpoint_dir, self._model_dir())
        os.makedirs(checkpoint_dir, exist_ok=True)
        if snapshot is None:
            snapshot = dict(params=self.params.detach().cpu(), m=self.m.cpu(), v=self.v.cpu(), t=self.step_counter.cpu().numpy())
        named = {TF_NAMES[k].replace("/", "__"): v.numpy() for k, v in self.named_params(snapshot["params"]).items()}
        path = os.path.join(checkpoint_dir, f"{model_name}-{step}.npz")
        np.savez(path, __flat__=np.asarray(snapshot["params"]), __variant__=np.int32(self.variant),
                 __adam_m__=np.asarray(snapshot["m"]), __adam_v__=np.asarray(snapshot["v"]),
                 __adam_t__=np.asarray(snapshot["t"]), **named)
        index = os.path.join(checkpoint_dir, "checkpoint")
        # max_to_keep = 5 is tracked IN MEMORY per model object, as tf.train.Saver does: files of an earlier run are
        # never deleted, and a name that is still among the last five is never removed (a rerun writes the same names)
        kept = self._saved.setdefault(checkpoint_dir, [])
        name = os.path.basename(path)
        if name in kept:
            kept.remove(name)
        kept.append(name)
        while len(kept) > 5:
            old = kept.pop(0)
            try:
                os.remove(os.path.join(checkpoint_dir, old))
            except OSError:
                pass
        with open(index, "w") as f:
            f.write("\n".join(kept) + "\n")
        return path

    def load(self, checkpoint_dir, note=None, restore_adam=False):
        if note is None:
            print(" [*] Reading checkpoint...")
        checkpoint_dir = os.path.join(checkpoint_dir, self._model_dir())
        index = os.path.join(checkpoint_dir, "checkpoint")
        if not os.path.exists(index):
            return False
        names = [l.strip() for l in open(index) if l.strip()]
        if not names:
            return False
        latest = os.path.join(checkpoint_dir, names[-1])
        if not os.path.exists(latest):
            return False
        z = np.load(latest)
        if int(z["__variant__"]) != self.variant or z["__flat__"].size != self.n_params:
            return False
        if note:
            print(note)
        self.params.copy_(torch.as_tensor(z["__flat__"]))
        if restore_adam:                                             # the reference never does (Q12)
            self.m.copy_(torch.as_tensor(z["__adam_m__"])); self.v.copy_(torch.as_tensor(z["__adam_v__"]))
            self.step_counter.copy_(torch.as_tensor(z["__adam_t__"]))
        return True
