#!/usr/bin/env python
"""bench.py -- training commits/s of the HD-GNN hot path on B200 (BASELINE.json metric).

A step = forward + backward + regularisers + TF-Adam over one batch of B synthetic commits per
GPU (model_2.py:369-383).  `value` times the step with inputs resident in HBM; `e2e` times the
public call `graph2graph.train_step` from pinned HOST buffers (H2D of the five compact inputs
and D2H of the loss inside the timed region).  `--impl reference` times the CPU restatement of
the reference (oracle/) on the host cores instead.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload glide|cfg2|cfg3|cfg4] [--variant 2] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {   # BASELINE.json configs; B = commits per GPU per step
    "glide": dict(Ne=200, Nc=74, B=100, step=2, desc="glide-shaped synthetic, Ne=200 Nc=74 Ner=39800 Ncr=5402"),
    "cfg2": dict(Ne=250, Nc=114, B=100, step=3, desc="synthetic Ne=250 Nc=114 Ner=62250 Ncr=12882 Step=3"),
    "cfg3": dict(Ne=250, Nc=150, B=100, step=5, desc="synthetic Ne=250 Nc=150 Ner=62250 Ncr=22350 Step=5"),
    "cfg4": dict(Ne=512, Nc=256, B=512, step=0, desc="synthetic scale-up Ne=512 Nc=256, 512 commits/GPU/step"),
}
L2_BYTES = 126 * 2 ** 20
METRIC = "train commits/sec (fwd+bwd+Adam)"
DUMP_BYTES = 64 * 10 ** 6      # --dump-outputs writes at most this much, .npy headers included


def write_outputs(out_dir, arrays):
    """arrays: name -> NumPy array, written as out_dir/<name>.npy in float32 (float arrays) or float64 (integer arrays).
    If they exceed DUMP_BYTES, `probs` keeps a fixed, seeded sample of its commits (rows), listed in probs_commits.npy."""
    arrays = {k: a.astype(np.float32 if a.dtype == np.float32 else np.float64, copy=False) for k, a in arrays.items()}
    p = arrays["probs"]
    rest = sum(a.nbytes for k, a in arrays.items() if k != "probs") + 4096      # + room for the headers
    if rest + p.nbytes > DUMP_BYTES:
        keep = (DUMP_BYTES - rest) // (p[0].nbytes + 8)
        rows = np.sort(np.random.default_rng(0).choice(p.shape[0], keep, replace=False))
        arrays["probs"], arrays["probs_commits"] = p[rows], rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def flops_fwd_per_commit(Ne, Nc, variant):
    """Canonical algorithmic FLOPs of the closed form, no one-hot matmuls, no collapse (SURVEY 8(d))."""
    ner, ncr = Ne * (Ne - 1), Nc * (Nc - 1)
    f = ncr * 2230 + ner * 8
    if variant in (2, 4):
        f += ner * 1000 + Ne * 880
    if variant == 4:
        f += ner * 1986
    return f


def bytes_per_commit_train(Ne, Nc):
    """Compulsory HBM bytes of one training step per commit in the u8 encoding: inputs read by
    forward and again by backward (recompute) + probs written (SURVEY 8(d))."""
    inp = Ne * Ne + 4 * Ne + 4 * Ne + 4 + Nc * Nc
    return 2 * inp + 8 * Nc * (Nc - 1)


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1]))
            except ValueError:
                continue
            for n, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_rate(Ne, Nc, variant, sample_commits, steps, warmup, dense=False):
    """fwd + bwd (autograd) + TF-Adam of the CPU restatement, fp32, all host threads.  dense=False: closed (index) form;
    dense=True: the literal one-hot matmuls the reference's TF graph executes (model_2.py:141-159).  Returns
    (commits/s from the MEDIAN step, cores, median seconds per step, (min, max) seconds)."""
    import torch
    from hdgnn_b200.synthetic import make_commits
    from oracle import hdgnn_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cb = make_commits(sample_commits, Ne, Nc, seed=20260)
    flat = O.init_params(variant, seed=1234, dtype=torch.float32)
    m = torch.zeros_like(flat); v = torch.zeros_like(flat)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        _, _, _, g, _ = O.train_loss_and_grad(variant, flat, cb.adj, cb.x, cb.hmap, cb.L, cb.Y, dense=dense)
        flat, m, v = O.tf_adam_step(flat, g, m, v, it + 1)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    med = float(np.median(times))
    return sample_commits / med, cores, med, (min(times), max(times))


def run_reference(args, wl, config):
    """--impl reference: the CPU restatement of the reference path on the host cores, on the SAME config as the GPU arm
    (same workload, same commits per step); K and W are honoured (3 warm-up steps at least, median step)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = args.ref_sample or wl["B"]
    rate, cores, sec, (tmin, tmax) = cpu_oracle_rate(wl["Ne"], wl["Nc"], args.variant, sample, args.steps, max(args.warmup, 3))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "commits/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config,
        "cpu_baseline": {"value": rate, "unit": "commits/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} commits/step x {args.steps} steps (median step; min {tmin * 1e3:.0f} ms, max {tmax * 1e3:.0f} ms) "
                                   "of the same workload; closed-form restatement of model_2.py:86-118 + autograd + TF-Adam in "
                                   "PyTorch-CPU fp32 (TensorFlow is not installable here, so the reference itself cannot run)"},
        "e2e": {"value": rate, "unit": "commits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def make_config(wl, variant, world):
    """The `config` object of the JSON line: identical for the GPU arm and the reference arm."""
    return {"workload": wl["desc"], "variant": variant, "commits_per_gpu_per_step": wl["B"], "global_batch": wl["B"] * world,
            "parallelism": f"dp{world} (commit-sharded)"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained"), "measured"
    return 6650.0, 1590.0, None, "fallback"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="glide", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", type=int, default=2)
    ap.add_argument("--batch", type=int, default=0, help="commits per GPU per step (default: workload's)")
    ap.add_argument("--ref-sample", type=int, default=0, help="commits per step of the CPU reference arm (default: the workload's B)")
    ap.add_argument("--repeats", type=int, default=1,
                    help="consecutive blocks the K timed steps are split into; the median block's time per step is reported")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (probabilities, losses, parameters, Adam state) as DIR/<name>.npy")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--loop-train", action="store_true", default=True, help="also time graph2graph.train() epochs (N=1)")
    ap.add_argument("--no-loop-train", dest="loop_train", action="store_false")
    ap.add_argument("--collective", default="auto", choices=["auto", "peer", "nccl"],
                    help="N>1 gradient exchange: fused into the last kernel over NVLink peer memory, or NCCL all-reduce")
    ap.add_argument("--rows-e", type=int, default=0)
    ap.add_argument("--rows-c", type=int, default=0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = dict(WORKLOADS[args.workload])
    if args.batch:
        wl["B"] = args.batch
    if args.warmup < 3:
        args.warmup = 3
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    config = make_config(wl, args.variant, world_env)
    if args.impl == "reference":
        return run_reference(args, wl, config)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"       # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from hdgnn_b200.engine import DeviceBatch
    from hdgnn_b200.model import graph2graph, HostBatch
    from hdgnn_b200.synthetic import make_commits

    Ne, Nc, B, variant = wl["Ne"], wl["Nc"], wl["B"], args.variant
    model = graph2graph(None, Ne=Ne, Nc=Nc, Mini_batch=B, Step=wl["step"], Repo="synthetic", variant=variant,
                        device=local, seed=1234, max_batch=B, collective=args.collective)
    eng = model.engine
    dev = eng.tdev
    # pool of distinct batches, larger than L2, generated globally (seed per pool slot and rank)
    batch_bytes = B * (Ne * eng.pe + Nc * eng.pc + 8 * Ne + 4)
    pool_n = max(4, int(np.ceil(1.25 * L2_BYTES / batch_bytes)) + 1)
    pool_n = min(pool_n, 256)
    n_distinct = min(pool_n, 32)        # distinct synthetic batches; further pool slots are copies at distinct addresses
    host_pool, dev_pool = [], []
    for i in range(pool_n):
        if i < n_distinct:
            cb = make_commits(B, Ne, Nc, seed=20260 + 1000 * rank + i)
        hb = model.host_batch(cb) if i < n_distinct else host_pool[i % n_distinct].clone()
        host_pool.append(hb)
        if i < n_distinct:
            dev_pool.append(DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, dev, bits=model.host_bits))
        else:
            d0 = dev_pool[i % n_distinct]
            dev_pool.append(DeviceBatch(d0.adj.clone(), d0.x.clone(), d0.hmap.clone(), d0.L.clone(), d0.Y.clone(), Ne, Nc))
    Bg = B * world
    probs = torch.empty(B, 2, eng.Ncr, dtype=torch.float32, device=dev)
    loss = torch.zeros(1, dtype=torch.float32, device=dev)

    loss3 = torch.zeros(3, dtype=torch.float32, device=dev)

    def device_step(k):
        db = dev_pool[k % pool_n]
        if world == 1:      # one fused call: forward, backward, gradient reduction + regularisers + Adam
            eng.train_step(db, model.params, model.m, model.v, model.step_counter, loss3, probs=probs)
            return eng.last_launch_count()
        if model.peer:      # same 5 launches: the all-reduce is fused into the reduce + Adam kernel (peer memory over NVLink)
            eng.train_step_peer(db, model.params, model.m, model.v, model.step_counter, loss3, probs=probs)
            return eng.last_launch_count()
        eng.forward_backward(db, model.params, B_global=Bg, grads=model.grads, probs=probs, loss=loss)
        n = eng.last_launch_count()
        dist.all_reduce(model.grads)
        eng.adam_step(model.params, model.grads, model.m, model.v, model.step_counter, reg_losses=model.reg)
        return n + eng.last_launch_count()

    def host_step(k):
        model.train_step(host_pool[k % pool_n])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def last_step_outputs():
        """What a caller of the timed step holds after its last step: probabilities, losses (CE, map MSE, parameter
        penalty; the CE is this rank's share on the multi-kernel path), the updated parameters and the Adam state."""
        torch.cuda.synchronize()
        losses = loss3 if world == 1 or model.peer else torch.cat([loss, model.reg])
        out = {"probs": probs, "losses": losses, "params": model.params, "adam_m": model.m, "adam_v": model.v,
               "adam_step": model.step_counter}
        return {k: t.detach().cpu().numpy() for k, t in out.items()}

    def timed(fn, steps, warmup, repeats, sample_clocks=False):
        """`warmup` untimed steps, then exactly `steps` timed steps in `repeats` consecutive blocks of (nearly) equal length,
        each bracketed by a barrier + synchronize on both sides and timed with CUDA events (max over ranks per block).
        Returns (milliseconds, steps) per block, launches of the timed steps, clocks."""
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler:         # the sampler's start-up wait comes before the warm-up, so the GPU is busy going into the timed steps
            sampler.start()
            time.sleep(0.15)
        for k in range(warmup):
            fn(k)
        barrier()
        blocks, launches, k0 = [], 0, warmup
        for n_steps in (len(a) for a in np.array_split(np.arange(steps), min(max(repeats, 1), steps))):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            for k in range(n_steps):
                launches += fn(k0 + k) or 0
            e1.record()
            barrier()
            k0 += n_steps
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            blocks.append((float(t.item()), n_steps))
        clocks = sampler.stop() if sampler else None
        return blocks, launches, clocks

    def per_step(blocks):
        return np.asarray([ms / n for ms, n in blocks])

    def spread(blocks):
        a = per_step(blocks)
        return {"blocks": len(blocks), "ms_per_step_median": float(np.median(a)), "ms_per_step_min": float(a.min()),
                "ms_per_step_max": float(a.max())}

    blocks_dev, launches, clocks = timed(device_step, args.steps, args.warmup, args.repeats, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, last_step_outputs())
    model.initialize(model.params.clone())      # reset Adam state, keep weights
    blocks_e2e, _, _ = timed(host_step, args.steps, args.warmup, args.repeats)
    ms_dev, ms_e2e = float(np.median(per_step(blocks_dev))), float(np.median(per_step(blocks_e2e)))     # per step
    value = Bg / (ms_dev * 1e-3)
    e2e_value = Bg / (ms_e2e * 1e-3)

    # the whole public loop: graph2graph.train() epochs (batch upload, step, accuracy counters, per-epoch log) on a
    # synthetic data set of 4 batches -- what `main.py --Type train` costs per step next to the bare step above
    loop = None
    if args.loop_train and world == 1:
        import types
        from hdgnn_b200.synthetic import CommitBatch
        nbat = 16
        parts = [make_commits(B, Ne, Nc, seed=777 + 1000 * rank + i) for i in range(nbat)]
        cat = CommitBatch(*[np.concatenate([getattr(c, f) for c in parts]) for f in ("adj", "x", "hmap", "L", "Y")])
        epochs = max(3, args.steps // nbat)
        keep = (model.epoch, model.mini_batch_num)
        model.epoch, model.mini_batch_num = epochs, B
        model.train(types.SimpleNamespace(Repo="bench", checkpoint_dir=""), data=(cat, None), quirk_q2=False, log=lambda *_: None,
                    save_checkpoints=False)
        torch.cuda.synchronize()
        dt = model.last_train_seconds            # the epoch loop as the reference times it (model_2.py:358,423): no data preparation
        model.epoch, model.mini_batch_num = keep
        if world == 1:
            loop = {"value": epochs * nbat * B / dt, "unit": "commits/s", "ms_per_step": dt * 1e3 / (epochs * nbat), "epochs": epochs,
                    "batches_per_epoch": nbat, "api": "graph2graph.train(): per step H2D of the batch and the fused step with the arg-max hit counter inside it; per epoch "
                    "an asynchronous snapshot of the parameters + hit count to pinned memory and the reference's log line, written "
                    "while the next epoch runs (no checkpoint files in this measurement)"}
        model.initialize(model.params.clone())

    # per-kernel timing pass (events around every launch; perturbs the step, so never the headline)
    eng.profile(True)
    prof_steps = min(args.steps, 20)
    for k in range(prof_steps):
        device_step(k)
    torch.cuda.synchronize()
    recs = eng.profile_records()
    eng.profile(False)
    agg = {}
    for name, ms in recs:
        a = agg.setdefault(name, [0.0, 0])
        a[0] += ms; a[1] += 1
    tot = sum(a[0] for a in agg.values())
    kernels = {n: {"avg_us": 1e3 * a[0] / a[1], "share": a[0] / tot} for n, a in agg.items()}
    top = max(agg, key=lambda n: agg[n][0])
    top_us = kernels[top]["avg_us"]
    ner, ncr = Ne * (Ne - 1), Nc * (Nc - 1)
    ent_inline = variant in (2, 4) and "ent_fwd" not in kernels and "pairsum_fwd(ent)" not in kernels
    alg = {   # canonical (un-collapsed) algorithmic FLOPs per launch of the reference ops each kernel covers (SURVEY 8(d) x pairs x B)
        "pairsum_fwd(ent)": B * ner * 1000, "pairsum_bwd(ent)": B * ner * 2000,
        "pairsum_fwd(edge)": B * ner * 1020, "pairsum_bwd(edge)": B * ner * 2040,
        "score_fwd(edge)": B * ner * 966, "score_bwd(edge)": B * ner * 3 * 966,
        "pairsum_fwd(hunk)": B * ncr * 1260, "pairsum_bwd(hunk)": B * ncr * 2520,
        "score(hunk)": B * ncr * 970 * 3,
        "ent_fwd": B * ner * 1000, "ent_bwd": B * ner * 2000,
        "mid(train)": B * 3 * (ncr * 2230 + ner * 8 + Ne * 880 + (ner * 1000 if ent_inline else 0)),
        "mid(infer)": B * (ncr * 2230 + ner * 8 + Ne * 880 + (ner * 1000 if ent_inline else 0)),
    }
    hbm_peak, bf16_peak, bf16_sus, src = measured_peaks()
    # denominators measured in THIS run: TF32 tensor throughput (cuBLAS through torch, 8192^3) and the fp32 CUDA-core peaks
    # (scalar FFMA and packed FFMA2 chains, hdgnn_measure_fp32_peak)
    peaks = {"hbm_gbs": hbm_peak, "bf16_tflops": bf16_peak, "source": f"MEASURED_PEAKS.json ({src})"}
    try:
        import ctypes as C
        from hdgnn_b200._lib import lib as L
        for name, packed in (("fp32_ffma_tflops", 0), ("fp32_ffma2_tflops", 1)):
            tf = C.c_float()
            if L.hdgnn_measure_fp32_peak(packed, C.byref(tf)) == 0:
                peaks[name] = tf.value
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        a32 = torch.randn(8192, 8192, device=dev); b32 = torch.randn(8192, 8192, device=dev)
        best = 0.0
        for _ in range(6):
            t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0e.record(); torch.matmul(a32, b32); t1e.record(); torch.cuda.synchronize()
            best = max(best, 2 * 8192 ** 3 / (t0e.elapsed_time(t1e) * 1e-3) / 1e12)
        torch.backends.cuda.matmul.allow_tf32 = old
        peaks["tf32_tflops"] = best
        del a32, b32
    except Exception as e:      # the peaks are diagnostics; the headline does not depend on them
        peaks["error"] = repr(e)
    tf32_peak = peaks.get("tf32_tflops") or bf16_peak / 2
    # Contract object for the dominant kernel.  The reference's pair layers are fp32 GEMMs, so the tensor bound is quoted
    # against the measured TF32 peak; `achieved` counts the CANONICAL flops of the reference formulation (no algebraic
    # collapse, SURVEY 8(d)) over the live kernel time.  The executed work is far smaller and runs on the CUDA cores
    # (DESIGN.md 3): `bounds` lists the same kernel against every ceiling that could apply, each with a measured peak.
    top_flops = alg.get(top, 0)
    top_bytes = B * bytes_per_commit_train(Ne, Nc)
    roof = {"kernel": top, "bound": "tensor", "unit": "TFLOP/s", "avg_us": top_us,
            "achieved": top_flops / (top_us * 1e-6) / 1e12, "peak": tf32_peak,
            "peak_source": "TF32 cuBLAS 8192^3 measured in this run (best of 6); achieved = canonical (un-collapsed) FLOPs of "
                           "SURVEY 8(d) / live kernel time, per launch of %d commits" % B,
            "traffic": None, "kernels": kernels, "peaks": peaks}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["bounds"] = [
        {"bound": "tensor (tf32)", "achieved": roof["achieved"], "peak": tf32_peak, "unit": "TFLOP/s", "frac": roof["frac"]},
        {"bound": "tensor (bf16 burst)", "achieved": roof["achieved"], "peak": bf16_peak, "unit": "TFLOP/s", "frac": roof["achieved"] / bf16_peak},
        {"bound": "fp32 CUDA cores (packed FFMA2)", "achieved": roof["achieved"], "peak": peaks.get("fp32_ffma2_tflops"), "unit": "TFLOP/s",
         "frac": roof["achieved"] / peaks["fp32_ffma2_tflops"] if peaks.get("fp32_ffma2_tflops") else None,
         "note": "canonical flops over the fp32 pipe's measured peak; above 1 means the collapsed algebra executes fewer flops than the reference formulation"},
        {"bound": "hbm", "achieved": top_bytes / (top_us * 1e-6) / 1e9, "peak": hbm_peak, "unit": "GB/s",
         "frac": top_bytes / (top_us * 1e-6) / 1e9 / hbm_peak, "note": "compulsory bytes of the u8 encoding (SURVEY 8(d)) per launch"},
    ]
    if "reduce_adam" in kernels:       # the optimizer kernel: B x P gradient partials in, 3 P floats in, 3 P out
        P = eng.n_params
        by = (B + 6) * P * 4
        roof["optimizer"] = {"kernel": "reduce_adam", "bound": "hbm (launch-latency in practice)", "avg_us": kernels["reduce_adam"]["avg_us"],
                             "achieved": by / (kernels["reduce_adam"]["avg_us"] * 1e-6) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": by / (kernels["reduce_adam"]["avg_us"] * 1e-6) / 1e9 / hbm_peak}
    try:        # DRAM traffic / executed instructions from the ncu capture of the same launch shape, only if it was taken on THIS library build
        import hashlib
        ic = json.load(open(os.path.join(ROOT, "profiles", "inst_counts.json")))
        from hdgnn_b200.build import LIB
        libhash = hashlib.sha256(open(LIB, "rb").read()).hexdigest()[:16]
        key = f"{args.workload}_B{B}_v{variant}"
        if ic.get("_lib_sha16") == libhash and top in ic.get(key, {}):
            roof["traffic"] = ic[key][top].get("dram_bytes")
            roof["ncu"] = {"lib_sha16": libhash, "kernels": ic[key]}
    except Exception:
        pass
    step_flops = 3 * flops_fwd_per_commit(Ne, Nc, variant)
    roof["step"] = {"algorithmic_tflops": value * step_flops / 1e12,
                    "algorithmic_hbm_gbs": value * bytes_per_commit_train(Ne, Nc) / 1e9,
                    "hbm_peak_gbs": hbm_peak, "hbm_frac": value * bytes_per_commit_train(Ne, Nc) / 1e9 / hbm_peak}

    # N > 1: the sharded step against one GPU on the same global batch (the driver's GPU test box has one GPU, so the
    # multi-GPU correctness check lives where N ranks actually run)
    parity = None
    if world > 1:
        parity = multi_gpu_parity(model, Ne, Nc, variant, world, rank, dev)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_sample = min(B, 100)
        rate, cores, sec, (tmin, tmax) = cpu_oracle_rate(Ne, Nc, variant, cpu_sample, 7, 3)
        cpu = {"value": rate, "unit": "commits/s", "cores": cores, "kind": "port",
               "sample": f"{cpu_sample} commits/step, 3 warm-up + 7 timed steps, median ({sec * 1e3:.0f} ms; min {tmin * 1e3:.0f}, max {tmax * 1e3:.0f}); "
                         "closed-form PyTorch-CPU fp32 restatement (oracle/hdgnn_oracle.py) incl. autograd backward and TF-Adam"}
        try:        # what the reference's TF graph literally executes: dense one-hot matmuls (model_2.py:141-159), small sample
            dn = 4 if Ne <= 256 else 1
            drate, _, dsec, _ = cpu_oracle_rate(Ne, Nc, variant, dn, 3, 1, dense=True)
            cpu["dense_leg"] = {"value": drate, "unit": "commits/s", "sample": f"{dn} commits/step, 1 warm-up + 3 timed steps, median ({dsec * 1e3:.0f} ms); "
                                "literal one-hot transcription (forward_dense) + autograd + TF-Adam"}
        except Exception as e:
            cpu["dense_leg"] = {"error": repr(e)}
    if rank == 0:
        config = make_config(wl, variant, world)         # identical to the reference arm's
        setup = {"collective": ("none" if world == 1 else
                                "gradient all-reduce fused into the reduce+Adam kernel over NVLink peer memory (no NCCL call in the step)"
                                if model.peer else "one NCCL gradient all-reduce/step between backward and Adam"),
                 "l2": f"inputs rotate through {pool_n} batch buffers ({n_distinct} distinct batches) = {pool_n * batch_bytes / 2**20:.0f} MiB > 126 MiB L2",
                 "entity_stage": ("inline (class tables / sorted prefix + edge walk)" if "ent_fwd" not in kernels and "pairsum_fwd(ent)" not in kernels
                                  else "dense sweeps") if variant in (2, 4) else "none",
                 # informational: what hdgnn.cu's fused_forward does for this shape (DESIGN.md section 5)
                 "per_commit_kernel": ("clusters of two CTAs, the costliest commits shared by both CTAs of a cluster"
                                       if (B < 148 and Nc <= 128 and variant != 4 and os.environ.get("HDGNN_CLUSTER", "1") != "0")
                                       else "one CTA per commit")}
        line = {
            "metric": METRIC, "value": value, "unit": "commits/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "setup": setup,
            "timing": {"device": spread(blocks_dev), "e2e": spread(blocks_e2e),
                       "note": f"{args.warmup} warm-up steps, then exactly {args.steps} timed steps in {len(blocks_dev)} block(s), each bracketed by "
                               "barrier + synchronize and timed with CUDA events (max over ranks); value / e2e are the MEDIAN block's time per step"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "commits/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": host_pool[0].nbytes(), "d2h_bytes_per_step": 12,
                    "wire_format": "label grids as bitmaps (HDGNN_F_LABEL_BITS), x f32, hmap i32, L i32" if model.host_bits else "label grids as u8",
                    "api": "hdgnn_b200.model.graph2graph.train_step: pinned host buffers -> hdgnn_train_step_host (1 GPU) / "
                           "hdgnn_train_step_peer_host (N GPUs, peer exchange) or hdgnn_forward_backward_host + NCCL all-reduce + hdgnn_adam_step; "
                           "H2D of step k+1 overlaps the kernels of step k",
                    "train_loop": loop},
            "gpu_launches": launches,
            "roofline": roof,
            "cpu_baseline": cpu,
        }
        if parity is not None:
            line["parity"] = parity
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def multi_gpu_parity(model, Ne, Nc, variant, world, rank, dev):
    """Three training steps of a fixed global batch on the sharded path (this run's collective), all ranks' parameters and
    Adam moments compared bitwise, and rank 0 repeating the same steps alone on the whole batch."""
    import torch
    import torch.distributed as dist
    from hdgnn_b200.engine import Engine, DeviceBatch, F_LABEL_BITS
    from hdgnn_b200.synthetic import make_commits
    from hdgnn_b200.model import truncated_normal_init
    per = min(8, model.max_batch)
    cbg = make_commits(per * world, Ne, Nc, seed=4242, p_short=0.5)
    flat = truncated_normal_init(variant, seed=99)
    model.initialize(flat.clone())
    hb = model.host_batch(cbg.slice(rank * per, (rank + 1) * per))
    for _ in range(3):
        model.train_step(hb)
    torch.cuda.synchronize()
    mine = torch.cat([model.params, model.m, model.v]).clone()
    allp = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allp, mine)
    identical = all(torch.equal(allp[0], t) for t in allp[1:])
    rel = None
    if rank == 0:
        bits = model.host_bits
        eng = Engine(Ne, Nc, variant=variant, max_batch=per * world, device=dev.index, flags=F_LABEL_BITS if bits else 0)
        db = DeviceBatch.from_numpy(cbg.adj, cbg.x, cbg.hmap, cbg.L, cbg.Y, dev, bits=bits)
        p = flat.to(dev).float(); m = torch.zeros_like(p); v = torch.zeros_like(p)
        step = torch.zeros(1, dtype=torch.int32, device=dev); loss3 = torch.zeros(3, device=dev)
        for _ in range(3):
            eng.train_step(db, p, m, v, step, loss3)
        torch.cuda.synchronize()
        rel = float((allp[0][:p.numel()] - p).abs().max() / p.abs().max())
        eng.close()
    model.initialize(flat.clone())
    return {"replicas_identical": bool(identical), "vs_single_gpu_rel": rel, "ranks": world,
            "what": f"3 Adam steps on a fixed global batch of {per * world} commits: params/m/v of all ranks compared bitwise; "
                    "rank 0's parameters vs one GPU training the whole batch (max abs diff / max abs)"}


if __name__ == "__main__":
    main()
