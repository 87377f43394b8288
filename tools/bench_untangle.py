"""Cost of the untangling output at Ne = 200, B = 100, Nc in {74, 256, 512} (variant 2, label bitmaps):
  (a) the device-resident forward writing the probabilities against the same forward writing only the predicted-relation
      bitmap (hdgnn_set_predictions, probs NULL);
  (b) host-fed inference end to end: probabilities copied to pinned host memory against predictions + hunk groups copied to
      pinned host memory (hdgnn_infer_host with probs NULL, then hdgnn_hunk_groups);
  (c) the hunk_groups kernel alone, on predicted and on label bitmaps;
  (d) the partition_counts kernel alone (the untangling scores) on the hunk groups of two label sets, every hunk real (the
      costliest case), at B = 100 and Nc in {74, 256, 512} and at B = 4096, Nc = 74, alternating with hunk_groups on the
      same commits; the per-call times of these eager blocks include the Python wrapper and the launch, so the kernel
      times are read from torch.profiler as well, in a pass of their own;
  (e) the hunk_clusters kernel alone (average linkage of the relation probabilities) at B = 100 and Nc in {74, 256, 512} and
      at B = 4096, Nc = 74, every hunk real, on planted groups of 8 hunks plus noise (nearly every merge happens: the costly
      case), alternating with hunk_groups on the arg-max bitmap of the same probabilities, kernel times from torch.profiler in
      a pass of their own; host-fed inference end to end as graph2graph.untangle runs it (Ne = 200, B = 100, random weights),
      grouping "average" (probabilities written to a device buffer, then hunk_clusters) against "components" (hunk_groups of
      the predicted relations); and the partition scores of both groupings against the planted groups when a few confident
      cross-group false positives are added;
  (f) the dendrogram: hunk_linkage (the whole merge sequence) against hunk_clusters at 0.5 on the same commits, at B = 100 and
      Nc in {74, 256, 512} and at B = 4096, Nc = 74, every hunk real, on planted groups of 8 and on random-weight
      probabilities (p1 ~ U(0, 1): the merges a threshold of 0.5 skips are many), and linkage_cut of the record at K = 1, 16
      and 64 thresholds, kernel times from torch.profiler in a pass per arm; and a sweep of 9 thresholds as
      graph2graph.untangle(sweep=...) runs it (one hunk_linkage, one linkage_cut, 9 partition_counts) against 9 hunk_clusters
      calls each followed by partition_counts, with the two arms' counters compared.
Device inputs rotate through copies that together exceed the 126 MB L2; every arm is timed in blocks that alternate with the
other arm's, and the median block is reported.  The card's name and power limit are read in the same run.
Usage: python tools/bench_untangle.py [--sections abcdef] [--out result.json]"""
import argparse, json, os, statistics, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from hdgnn_b200.EvaluationFuncs import partition_metrics_from_counts
from hdgnn_b200._lib import lib
from hdgnn_b200.engine import (Engine, DeviceBatch, F_LABEL_BITS, bit_words, hunk_clusters, hunk_groups, hunk_linkage,
                               linkage_cut, pack_label_bits, partition_counts)
from hdgnn_b200.model import HostBatch
from hdgnn_b200.synthetic import make_commits

L2_BYTES = 126 << 20
B, Ne, REPS = 100, 200, 9


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"nvidia_smi": q[torch.cuda.current_device()] if q else None, "torch_name": torch.cuda.get_device_name()}


def rotate(tensors, nbytes):
    """Enough device copies of a list of batches that one pass over them reads more than the L2 holds."""
    copies = max(len(tensors), -(-2 * L2_BYTES // max(nbytes, 1)))
    return [tensors[i % len(tensors)].clone() if torch.is_tensor(tensors[i % len(tensors)]) else
            DeviceBatch(*(getattr(tensors[i % len(tensors)], k).clone() for k in ("adj", "x", "hmap", "L", "Y")), Ne=tensors[0].Ne,
                        Nc=tensors[0].Nc) for i in range(copies)]


def timed(arms, calls):
    """{name: median ms per call} over REPS blocks of `calls` calls, the arms alternating block by block."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    got = {k: [] for k in arms}
    for name, fn in arms.items():          # warm-up of every arm
        for k in range(3):
            fn(k)
    torch.cuda.synchronize()
    for r in range(REPS):
        for name, fn in arms.items():
            e0.record()
            for k in range(calls):
                fn(r * calls + k)
            e1.record()
            torch.cuda.synchronize()
            got[name].append(e0.elapsed_time(e1) / calls)
    return {k: statistics.median(v) for k, v in got.items()}, got


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sections", default="abcdef", help="which of the sections (a)-(f) to run")
    args = ap.parse_args()
    out = {"card": card(), "B": B, "Ne": Ne, "variant": 2, "reps": REPS, "what": __doc__.split("Usage")[0].strip(), "rows": []}
    for Nc in ((74, 256, 512) if set("abc") & set(args.sections) else ()):
        eng = Engine(Ne, Nc, variant=2, max_batch=B, flags=F_LABEL_BITS)
        WPc = bit_words(Nc)
        cbs = [make_commits(B, Ne, Nc, seed=4040 + i) for i in range(4)]
        dbs = [DeviceBatch.from_numpy(c.adj, c.x, c.hmap, c.L, c.Y, eng.tdev, bits=True) for c in cbs]
        per_batch = sum(t.numel() * t.element_size() for t in (dbs[0].adj, dbs[0].x, dbs[0].hmap, dbs[0].L, dbs[0].Y))
        pool = rotate(dbs, per_batch)
        g = torch.Generator().manual_seed(1)
        params = (0.1 * torch.randn(eng.n_params, generator=g)).cuda()
        pred = torch.zeros(B, Nc, WPc, dtype=torch.int32, device="cuda")
        row = {"Nc": Nc, "device_pool_batches": len(pool)}

        # (a) device-resident forward
        def fwd_probs(k):
            eng.forward(pool[k % len(pool)], params, want_logits=False)

        def fwd_pred(k):
            eng.forward(pool[k % len(pool)], params, want_logits=False, want_probs=False)
        blocks_a = {"probs": [], "pred": []}
        for r in range(REPS):
            eng.set_predictions(None)
            m1, _ = timed_once(fwd_probs, r, 20)
            eng.set_predictions(pred)
            m2, _ = timed_once(fwd_pred, r, 20)
            blocks_a["probs"].append(m1); blocks_a["pred"].append(m2)
        eng.set_predictions(None)
        ms_a = {k: statistics.median(v) for k, v in blocks_a.items()}
        row["a_device_forward"] = {"ms_per_batch_probs": ms_a["probs"], "ms_per_batch_pred_only": ms_a["pred"],
                                   "commits_per_s_probs": B / ms_a["probs"] * 1e3, "commits_per_s_pred_only": B / ms_a["pred"] * 1e3,
                                   "blocks_ms": blocks_a}

        # (b) host-fed inference end to end
        hbs = [HostBatch(c, bits=True) for c in cbs]
        probs_h = torch.empty(B, 2, Nc * (Nc - 1), dtype=torch.float32).pin_memory()
        pred_h = torch.empty(B, Nc, WPc, dtype=torch.int32).pin_memory()
        groups_h = torch.empty(B, Nc, dtype=torch.int32).pin_memory()
        loss_h = torch.empty(1, dtype=torch.float32).pin_memory()

        def host_probs(k):
            eng.infer_host(*hbs[k % len(hbs)].tensors(), params, probs_h, loss_h)

        def host_groups(k):
            eng.infer_host(*hbs[k % len(hbs)].tensors(), params, None, loss_h)
            gr, _ = hunk_groups(pred)
            pred_h.copy_(pred, non_blocking=True)
            groups_h.copy_(gr, non_blocking=True)
        calls = 10 if Nc >= 256 else 40
        blocks_b = {"probs": [], "pred_groups": []}
        for r in range(REPS):
            eng.set_predictions(None)
            blocks_b["probs"].append(timed_once(host_probs, r, calls)[0])
            eng.set_predictions(pred)
            blocks_b["pred_groups"].append(timed_once(host_groups, r, calls)[0])
        eng.set_predictions(None)
        ms_b = {k: statistics.median(v) for k, v in blocks_b.items()}
        row["b_host_fed"] = {"ms_per_batch_probs_to_host": ms_b["probs"], "ms_per_batch_pred_groups_to_host": ms_b["pred_groups"],
                             "commits_per_s_probs_to_host": B / ms_b["probs"] * 1e3,
                             "commits_per_s_pred_groups_to_host": B / ms_b["pred_groups"] * 1e3,
                             "probs_bytes_per_batch": probs_h.numel() * 4,
                             "pred_groups_bytes_per_batch": pred_h.numel() * 4 + groups_h.numel() * 4, "blocks_ms": blocks_b}

        # (c) hunk_groups alone, on predicted and on label bitmaps
        preds = []
        eng.set_predictions(pred)
        for db in dbs:
            eng.forward(db, params, want_logits=False, want_probs=False)
            preds.append(pred.clone())
        eng.set_predictions(None)
        bitmap_bytes = B * Nc * WPc * 4
        pred_pool = rotate(preds, bitmap_bytes)
        lab_pool = rotate([db.Y for db in dbs], bitmap_bytes)
        ms_c, blocks_c = timed({"pred": lambda k: hunk_groups(pred_pool[k % len(pred_pool)]),
                                "labels": lambda k: hunk_groups(lab_pool[k % len(lab_pool)])}, 50)
        ng_pred = float(hunk_groups(pred_pool[0])[1].float().mean())
        ng_lab = float(hunk_groups(lab_pool[0])[1].float().mean())
        row["c_hunk_groups"] = {"us_per_batch_pred": ms_c["pred"] * 1e3, "us_per_batch_labels": ms_c["labels"] * 1e3,
                                "commits_per_s_pred": B / ms_c["pred"] * 1e3, "commits_per_s_labels": B / ms_c["labels"] * 1e3,
                                "mean_groups_pred": ng_pred, "mean_groups_labels": ng_lab, "bitmap_pool_batches": len(pred_pool),
                                "blocks_ms": blocks_c}
        print(json.dumps({k: v for k, v in row.items()}, default=str))
        out["rows"].append(row)
        del pool, pred_pool, lab_pool
        eng.close()
        torch.cuda.empty_cache()
    if "d" in args.sections:
        out["d_partition_counts"] = [scores(Bd, Nc) for Bd, Nc in ((B, 74), (B, 256), (B, 512), (4096, 74))]
    if "e" in args.sections:
        out["e_hunk_clusters"] = [clusters(Bd, Nc) for Bd, Nc in ((B, 74), (B, 256), (B, 512), (4096, 74))]
        out["e_untangle_end_to_end"] = [untangle_e2e(Nc) for Nc in (74, 256, 512)]
        out["e_quality"] = [quality(Nc) for Nc in (74, 256)]
    if "f" in args.sections:
        out["f_linkage"] = [linkage_row(Bd, Nc, kind) for Bd, Nc in ((B, 74), (B, 256), (B, 512), (4096, 74))
                            for kind in ("planted", "random")]
        out["f_sweep"] = [sweep_row(Nc) for Nc in (74, 256, 512)]
    out["card_after"] = card()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(out, open(args.out, "w"), indent=1)


def scores(Bd, Nc):
    """(d): partition_counts of two groupings of Bd commits (the hunk groups of two synthetic label sets, nh = Nc), in blocks
    alternating with hunk_groups of the first label set."""
    lab = [torch.as_tensor(pack_label_bits(make_commits(Bd, 8, Nc, seed=5050 + i, p_noise=1.0 / Nc).Y).view(np.int32)).cuda()
           for i in range(2)]
    groups = [hunk_groups(x)[0] for x in lab]
    nh = torch.full((Bd,), Nc, dtype=torch.int32, device="cuda")
    pairs = rotate([torch.stack(groups)], 2 * Bd * Nc * 4)
    bits = rotate([lab[0]], lab[0].numel() * 4)
    ms, blocks = timed({"partition_counts": lambda k: partition_counts(pairs[k % len(pairs)][0], pairs[k % len(pairs)][1], nh),
                        "hunk_groups": lambda k: hunk_groups(bits[k % len(bits)])}, 50)
    kern = kernel_us({"partition_counts": lambda k: partition_counts(pairs[k % len(pairs)][0], pairs[k % len(pairs)][1], nh),
                      "hunk_groups": lambda k: hunk_groups(bits[k % len(bits)])}, 200)
    c = partition_counts(groups[0], groups[1], nh).cpu().numpy()
    row = {"B": Bd, "Nc": Nc, "us_per_batch_partition_counts": ms["partition_counts"] * 1e3,
           "us_per_batch_hunk_groups": ms["hunk_groups"] * 1e3, "commits_per_s_partition_counts": Bd / ms["partition_counts"] * 1e3,
           "kernel_us_partition_counts": kern.get("partition_counts"), "kernel_us_hunk_groups": kern.get("hunk_groups"),
           "mean_groups": [float(c[:, 4].mean()), float(c[:, 5].mean())], "pool_batches": len(pairs), "blocks_ms": blocks}
    print(json.dumps(row, default=str))
    return row


def planted(Bd, Nc, seed, group=8, p_false=0.0):
    """(probs (Bd, 2, Nc(Nc-1)) f32, truth (Bd, Nc) int32) on the device: each commit's hunks in random groups of `group`;
    p1 ~ U(0.55, 0.95) inside a group (15 % of the inner pairs missing at U(0, 0.3)), U(0, 0.35) across, plus a fraction
    p_false of the cross pairs at U(0.8, 1); both directions drawn on their own; p0 = 1 - p1.  truth = the smallest hunk of
    each hunk's planted group."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = lambda lo, hi: lo + (hi - lo) * torch.rand(Bd, Nc, Nc, generator=g, device="cuda")
    lab = torch.argsort(torch.rand(Bd, Nc, generator=g, device="cuda"), dim=1) // group
    same = lab[:, :, None] == lab[:, None, :]
    P = torch.where(same, u(0.55, 0.95), u(0.0, 0.35))
    P = torch.where(same & (torch.rand(Bd, Nc, Nc, generator=g, device="cuda") < 0.15), u(0.0, 0.3), P)
    P = torch.where(~same & (torch.rand(Bd, Nc, Nc, generator=g, device="cuda") < p_false), u(0.8, 1.0), P)
    off = ~torch.eye(Nc, dtype=torch.bool, device="cuda")
    p1 = P[:, off]                                   # row-major without the diagonal: the pair order s(Nc-1)+t-[t>s]
    probs = torch.stack([1 - p1, p1], dim=1).contiguous()
    idx = torch.arange(Nc, device="cuda").expand(Bd, Nc)
    first = torch.full((Bd, Nc), Nc, dtype=torch.int64, device="cuda").scatter_reduce(1, lab, idx, "amin")
    return probs, torch.gather(first, 1, lab).to(torch.int32)


def argmax_bits(probs, Nc):
    p = probs.cpu().numpy()
    grid = np.zeros((p.shape[0], Nc, Nc), dtype=np.uint8)
    grid[:, ~np.eye(Nc, dtype=bool)] = p[:, 1] > p[:, 0]
    return torch.as_tensor(pack_label_bits(grid).view(np.int32)).cuda()


def clusters(Bd, Nc):
    """(e): hunk_clusters of Bd commits (every hunk real, planted groups of 8), in blocks alternating with hunk_groups of the
    arg-max bitmap of the same probabilities."""
    probs, _ = planted(Bd, Nc, 6060)
    bits = argmax_bits(probs, Nc)
    nh = torch.full((Bd,), Nc, dtype=torch.int32, device="cuda")
    ppool = rotate([probs], probs.numel() * 4)
    bpool = rotate([bits], bits.numel() * 4)
    arms = {"hunk_clusters": lambda k: hunk_clusters(ppool[k % len(ppool)], nh, 0.5),
            "hunk_groups": lambda k: hunk_groups(bpool[k % len(bpool)])}
    calls = 5 if Nc >= 256 else 20
    ms, blocks = timed(arms, calls)
    kern = kernel_us(arms, 4 * calls)
    ng_avg = hunk_clusters(probs, nh, 0.5)[1].float().mean().item()
    ng_cc = hunk_groups(bits)[1].float().mean().item()
    row = {"B": Bd, "Nc": Nc, "us_per_batch_hunk_clusters": ms["hunk_clusters"] * 1e3, "us_per_batch_hunk_groups": ms["hunk_groups"] * 1e3,
           "commits_per_s_hunk_clusters": Bd / ms["hunk_clusters"] * 1e3,
           "kernel_us_hunk_clusters": kern.get("hunk_clusters"), "kernel_us_hunk_groups": kern.get("hunk_groups"),
           "merges_per_commit": Nc - ng_avg, "mean_groups_average": ng_avg, "mean_groups_components": ng_cc,
           "work_bytes": int(lib.hdgnn_hunk_clusters_work(Bd, Nc)),
           "pool_batches": len(ppool), "blocks_ms": blocks}
    print(json.dumps(row, default=str))
    del ppool, bpool
    torch.cuda.empty_cache()
    return row


def untangle_e2e(Nc):
    """(e): host-fed inference + groups per batch as graph2graph.untangle runs it, "average" against "components"."""
    eng = Engine(Ne, Nc, variant=2, max_batch=B, flags=F_LABEL_BITS)
    cbs = [make_commits(B, Ne, Nc, seed=7070 + i) for i in range(4)]
    hbs = [HostBatch(c, bits=True) for c in cbs]
    params = (0.1 * torch.randn(eng.n_params, generator=torch.Generator().manual_seed(1))).cuda()
    pred = torch.zeros(B, Nc, bit_words(Nc), dtype=torch.int32, device="cuda")
    probs = torch.empty(B, 2, Nc * (Nc - 1), dtype=torch.float32, device="cuda")
    nh = torch.full((B,), Nc, dtype=torch.int32, device="cuda")
    groups = torch.empty(B, Nc, dtype=torch.int32, device="cuda")
    eng.set_predictions(pred)

    def average(k):
        eng.infer_host(*hbs[k % len(hbs)].tensors(), params, probs, None)
        groups.copy_(hunk_clusters(probs, nh, 0.5)[0])

    def components(k):
        eng.infer_host(*hbs[k % len(hbs)].tensors(), params, None, None)
        groups.copy_(hunk_groups(pred)[0])
    ms, blocks = timed({"average": average, "components": components}, 5 if Nc >= 256 else 20)
    ng = hunk_clusters(probs, nh, 0.5)[1].float().mean().item()
    eng.set_predictions(None)
    eng.close()
    row = {"Nc": Nc, "B": B, "Ne": Ne, "ms_per_batch_average": ms["average"], "ms_per_batch_components": ms["components"],
           "commits_per_s_average": B / ms["average"] * 1e3, "commits_per_s_components": B / ms["components"] * 1e3,
           "mean_groups_average_random_weights": ng, "blocks_ms": blocks}
    print(json.dumps(row, default=str))
    return row


def quality(Nc, Bq=200):
    """(e): partition scores against the planted groups of both groupings, on planted probabilities with 1 % of the cross pairs
    confident false positives."""
    probs, truth = planted(Bq, Nc, 8080, p_false=0.01)
    nh = torch.full((Bq,), Nc, dtype=torch.int32, device="cuda")
    avg = hunk_clusters(probs, nh, 0.5)[0]
    cc = hunk_groups(argmax_bits(probs, Nc))[0]
    row = {"Nc": Nc, "B": Bq, "p_false": 0.01, "group": 8,
           "average": partition_metrics_from_counts(partition_counts(avg, truth, nh).cpu().numpy()),
           "components": partition_metrics_from_counts(partition_counts(cc, truth, nh).cpu().numpy())}
    print(json.dumps(row, default=str))
    return row


def random_probs(Bd, Nc, seed):
    """(Bd, 2, Nc(Nc-1)) f32 on the device: p1 ~ U(0, 1) for every pair, p0 = 1 - p1 (a forward with random weights is
    about as unstructured)."""
    p1 = torch.rand(Bd, Nc * (Nc - 1), generator=torch.Generator(device="cuda").manual_seed(seed), device="cuda")
    return torch.stack([1 - p1, p1], dim=1).contiguous()


# kernel of each arm of section (f): the threshold and the recording instantiation of hunk_clusters_kernel share a name
F_KERNELS = {"hunk_clusters": ("hunk_clusters_kernel", ("<false>", "ILb0E")), "hunk_linkage": ("hunk_clusters_kernel", ("<true>", "ILb1E")),
             "cut_K1": ("linkage_cut_kernel", ("",)), "cut_K16": ("linkage_cut_kernel", ("",)), "cut_K64": ("linkage_cut_kernel", ("",))}


def kernel_us_each(arms, calls):
    """{arm: mean device time in µs of its kernel (F_KERNELS)}, one torch.profiler pass per arm."""
    from torch.profiler import profile, ProfilerActivity
    got = {}
    for name, fn in arms.items():
        kern, tags = F_KERNELS[name]
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for k in range(calls):
                fn(k)
            torch.cuda.synchronize()
        for e in prof.key_averages():
            if kern in e.key and any(t in e.key for t in tags) and e.count:
                got[name] = e.device_time_total / e.count
    return got


def linkage_row(Bd, Nc, kind):
    """(f): hunk_linkage against hunk_clusters(0.5), and linkage_cut at K = 1, 16, 64, on the same Bd commits."""
    probs = planted(Bd, Nc, 6161)[0] if kind == "planted" else random_probs(Bd, Nc, 6161)
    nh = torch.full((Bd,), Nc, dtype=torch.int32, device="cuda")
    rec = hunk_linkage(probs, nh)
    ppool = rotate([probs], probs.numel() * 4)
    rbytes = sum(x.numel() * 4 for x in rec)
    rpool = [tuple(x.clone() for x in rec) for _ in range(max(1, -(-2 * L2_BYTES // rbytes)))]
    ts = [float(t) for t in np.linspace(0.05, 0.95, 64)]
    arms = {"hunk_clusters": lambda k: hunk_clusters(ppool[k % len(ppool)], nh, 0.5),
            "hunk_linkage": lambda k: hunk_linkage(ppool[k % len(ppool)], nh)}
    for K in (1, 16, 64):
        arms[f"cut_K{K}"] = (lambda K: lambda k: linkage_cut(*rpool[k % len(rpool)], nh, thresholds=ts[:K]))(K)
    calls = 5 if Nc >= 256 else 20
    ms, blocks = timed(arms, calls)
    kern = kernel_us_each(arms, 4 * calls)
    g, ng = linkage_cut(*rec, nh, thresholds=[0.5])
    gc, ngc = hunk_clusters(probs, nh, 0.5)
    row = {"B": Bd, "Nc": Nc, "probs": kind, **{f"us_per_call_{k}": v * 1e3 for k, v in ms.items()},
           **{f"kernel_us_{k}": kern.get(k) for k in arms},
           "merges_per_commit_linkage": float(rec[2].float().mean()), "merges_per_commit_clusters_0.5": Nc - float(ngc.float().mean()),
           "cut_0.5_equals_hunk_clusters": bool(torch.equal(g[0], gc) and torch.equal(ng[0], ngc)),
           "pool_batches": len(ppool), "record_pool_batches": len(rpool), "blocks_ms": blocks}
    print(json.dumps(row, default=str))
    del ppool, rpool
    torch.cuda.empty_cache()
    return row


def sweep_row(Nc, Bd=B):
    """(f): 9 thresholds scored as graph2graph.untangle(sweep=...) does it, against 9 hunk_clusters + partition_counts."""
    probs, truth = planted(Bd, Nc, 6262, p_false=0.01)
    nh = torch.full((Bd,), Nc, dtype=torch.int32, device="cuda")
    ppool = rotate([probs], probs.numel() * 4)
    ts = [0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9]
    counts = torch.empty(2, len(ts), Bd, 8, dtype=torch.int64, device="cuda")

    def linkage_sweep(k):
        p = ppool[k % len(ppool)]
        g = linkage_cut(*hunk_linkage(p, nh), nh, thresholds=ts)[0]
        for i in range(len(ts)):
            counts[0, i] = partition_counts(g[i], truth, nh)

    def clusters_x9(k):
        p = ppool[k % len(ppool)]
        for i, t in enumerate(ts):
            counts[1, i] = partition_counts(hunk_clusters(p, nh, t)[0], truth, nh)
    ms, blocks = timed({"linkage_sweep": linkage_sweep, "clusters_x9": clusters_x9}, 2 if Nc >= 256 else 5)
    linkage_sweep(0)
    clusters_x9(0)
    row = {"B": Bd, "Nc": Nc, "thresholds": ts, "ms_per_batch_linkage_sweep": ms["linkage_sweep"],
           "ms_per_batch_9_hunk_clusters": ms["clusters_x9"], "counts_equal": bool(torch.equal(counts[0], counts[1])),
           "pair_f1": [partition_metrics_from_counts(counts[0, i].cpu().numpy())["pair_f1"] for i in range(len(ts))],
           "ari": [partition_metrics_from_counts(counts[0, i].cpu().numpy())["ari"] for i in range(len(ts))],
           "pool_batches": len(ppool), "blocks_ms": blocks}
    print(json.dumps(row, default=str))
    del ppool
    torch.cuda.empty_cache()
    return row


def kernel_us(arms, calls):
    """{name: mean device time in µs of the kernel `{name}_kernel`} over `calls` calls of each arm, from torch.profiler."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for fn in arms.values():
            for k in range(calls):
                fn(k)
        torch.cuda.synchronize()
    got = {}
    for e in prof.key_averages():
        for name in arms:
            if f"{name}_kernel" in e.key and e.count:
                got[name] = e.device_time_total / e.count
    return got


def timed_once(fn, r, calls):
    """ms per call of one block of `calls` calls (ends in a device synchronise)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn(r * calls)
    torch.cuda.synchronize()
    e0.record()
    for k in range(calls):
        fn(r * calls + k)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls, None


if __name__ == "__main__":
    main()
