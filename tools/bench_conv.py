"""Achieved HBM bandwidth of the legacy operator kernels (k_conv.cu): bytes = adjacency tile + H/x in + out.

--format bytes (default): byte grids, 3 warm-up and 10 timed calls per entry point, one line per entry point and shape.
--format bits: the same on label bitmaps (HDGNN_P_LABEL_BITS).
--format both: byte grids and label bitmaps of the same adjacency, timed in alternating blocks in one process.  A bitmap
  working set fits the 126 MB L2 (29 MB for map_conv at B = 4096), so every block rotates over copies of all inputs that
  together exceed twice the L2: a call never finds its inputs left in L2 by the call before.  The JSON records the GPU and
  its power limit beside the numbers.
"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from hdgnn_b200.engine import (normalize_propagate, map_conv, normalize_propagate_backward, map_conv_backward, label_pitch,
                               bit_words, pack_label_bits_device)

ap = argparse.ArgumentParser()
ap.add_argument("--format", choices=("bytes", "bits", "both"), default="bytes")
ap.add_argument("--blocks", type=int, default=7, help="--format both: timed blocks per format and entry point")
ap.add_argument("--calls", type=int, default=40, help="--format both: calls per timed block")
ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
args = ap.parse_args()

peak = 6543.4
try:
    peak = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")))["hbm_gbs"]
except Exception:
    pass
L2_BYTES = 126 << 20
SHAPES = [(4096, 200, 1, 0.05), (4096, 200, 20, 0.05), (4096, 200, 20, 0.5), (2048, 250, 20, 0.05)]


def entry_points(adj, x, H, theta, dOut, B, N, d, row_bytes):
    """(name, call, bytes moved) of the entry points timed at this shape; row_bytes = the adjacency row of the format."""
    eps = [("map_conv", lambda a, x, H, dO: map_conv(a, x, theta), B * (N * row_bytes + 4 * N + 4)),
           ("map_conv_backward", lambda a, x, H, dO: map_conv_backward(a, x, theta), B * (N * row_bytes + 8 * N + 8)),
           (f"normalize_propagate d={d}", lambda a, x, H, dO: normalize_propagate(a, H), B * (N * row_bytes + 8 * N * d + 4 * N)),
           (f"normalize_propagate_backward d={d}", lambda a, x, H, dO: normalize_propagate_backward(a, H, dO),
            B * (N * row_bytes + 12 * N * d))]
    return [e for e in eps if e[0].startswith("map_conv") == (d == 1)]


def gpu_identity():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = float(q.stdout.strip().splitlines()[0])
    except Exception:
        power = None
    return name, power


def time_block(fn, sets, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(20_000_000)          # lets the host queue the block ahead of the GPU
    e0.record()
    for k in range(calls):
        fn(*sets[k % len(sets)])
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


res = []
for (B, N, d, p) in SHAPES:
    pitch = label_pitch(N)
    g = torch.Generator(device="cuda").manual_seed(1)
    adj = (torch.rand(B, N, pitch, device="cuda", generator=g) < p).to(torch.uint8)
    adj[:, :, N:] = 0
    x = torch.rand(B, N, device="cuda", generator=g)
    H = torch.rand(B, N, d, device="cuda", generator=g)
    theta = torch.tensor([0.1, -0.2], device="cuda")
    dOut = torch.rand(B, N, d, device="cuda", generator=g)
    if args.format != "both":
        a = adj if args.format == "bytes" else pack_label_bits_device(adj)
        row = pitch if args.format == "bytes" else 4 * bit_words(N)
        for name, fn, nbytes in entry_points(a, x, H, theta, dOut, B, N, d, row):
            for _ in range(3):
                fn(a, x, H, dOut)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                fn(a, x, H, dOut)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 10
            gbs = nbytes / ms / 1e6
            res.append({"kernel": name, "B": B, "N": N, "density": p, "ms": ms, "GB/s": gbs, "frac_of_measured_hbm_peak": gbs / peak})
            if args.format == "bits":
                res[-1]["format"] = "bits"
            print(res[-1])
        continue
    bits = pack_label_bits_device(adj)
    fmts = {"bytes": (adj, pitch), "bits": (bits, 4 * bit_words(N))}
    for i, (name, _, _) in enumerate(entry_points(adj, x, H, theta, dOut, B, N, d, pitch)):
        row = {"kernel": name, "B": B, "N": N, "density": p}
        sets, calls = {}, {}
        for f, (a, rb) in fmts.items():
            _, fn, nbytes = entry_points(a, x, H, theta, dOut, B, N, d, rb)[i]
            # copies of every input the call reads, rotated so that the set of copies exceeds twice the L2
            ncopy = max(2, -(-2 * L2_BYTES // nbytes))
            sets[f] = [(a.clone(), x.clone(), H.clone(), dOut.clone()) for _ in range(ncopy)]
            calls[f] = (fn, nbytes, ncopy)
            for s in sets[f]:
                fn(*s)
        torch.cuda.synchronize()
        times = {f: [] for f in fmts}
        for _ in range(args.blocks):
            for f in fmts:
                times[f].append(time_block(calls[f][0], sets[f], args.calls))
        for f in fmts:
            ms = float(np.median(times[f]))
            gbs = calls[f][1] / ms / 1e6
            row[f] = {"ms": ms, "ms_blocks": times[f], "bytes_per_call": calls[f][1], "GB/s": gbs,
                      "frac_of_measured_hbm_peak": gbs / peak, "input_copies": calls[f][2]}
        row["bits_over_bytes_time"] = row["bits"]["ms"] / row["bytes"]["ms"]
        res.append(row)
        print(json.dumps({k: v for k, v in row.items()}, default=float))
        del sets
        torch.cuda.empty_cache()
if args.format == "both":
    name, power = gpu_identity()
    res = {"gpu": name, "power_limit_w": power, "hbm_peak_gbs_used": peak,
           "l2": "inputs rotated over copies totalling more than 2 x 126 MB in every timed block",
           "timing": f"median over {args.blocks} alternating blocks of {args.calls} back-to-back calls, CUDA events",
           "results": res}
if args.out:
    json.dump(res, open(args.out, "w"), indent=1)
