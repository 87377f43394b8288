"""BASELINE.json config 5: inference-only sweep (--Type test path), Ne = 200, Nc 74 -> 512, B = 100.
Prints commits/s and hunk pairs/s for the device-resident forward (hdgnn_forward, probs only)."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from hdgnn_b200.engine import Engine, DeviceBatch, F_LABEL_BITS, eval_counts
from hdgnn_b200.synthetic import make_commits

B, Ne = 100, 200
out = []
for Nc in (74, 114, 150, 256, 384, 512):
    eng = Engine(Ne, Nc, variant=2, max_batch=B, flags=F_LABEL_BITS)      # label bitmaps resident in HBM
    pool, ybytes = [], []
    for i in range(8):
        cb = make_commits(B, Ne, Nc, seed=20260 + i)
        pool.append(DeviceBatch.from_numpy(cb.adj, cb.x, cb.hmap, cb.L, cb.Y, eng.tdev, bits=eng.host_bits))
        ybytes.append(torch.as_tensor(cb.Y).cuda())
    params = (0.1 * torch.randn(eng.n_params)).cuda()
    for k in range(5):
        eng.forward(pool[k % 8], params, want_logits=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 50
    e0.record()
    for k in range(steps):
        eng.forward(pool[k % 8], params, want_logits=False)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    # the same with the evaluation counters (top_ACC / P / R / F1) computed on the device after every batch
    e0.record()
    for k in range(steps):
        probs, _, _ = eng.forward(pool[k % 8], params, want_logits=False)
        eval_counts(probs, ybytes[k % 8])
    e1.record(); torch.cuda.synchronize()
    ms_eval = e0.elapsed_time(e1) / steps
    # ... and with the counters taken inside the relation head (hdgnn_set_eval_counters): what graph2graph.test() does
    counts = torch.zeros(B, 8, dtype=torch.int64, device="cuda")
    ms_evk = None
    if eng.set_eval_counters(counts):
        eng.forward(pool[0], params, want_logits=False)
        e0.record()
        for k in range(steps):
            eng.forward(pool[k % 8], params, want_logits=False)
        e1.record(); torch.cuda.synchronize()
        ms_evk = e0.elapsed_time(e1) / steps
        eng.set_eval_counters(None)
    rec = {"label_bits": eng.host_bits, "ms_per_batch_with_eval": ms_eval, "ms_per_batch_with_in_kernel_counters": ms_evk,"Ne": Ne, "Nc": Nc, "B": B, "ms_per_batch": ms, "commits_per_s": B / ms * 1e3,
           "hunk_pairs_per_s": B * Nc * (Nc - 1) / ms * 1e3, "launches": eng.last_launch_count(),
           "probs_GBps": B * 8 * Nc * (Nc - 1) / ms / 1e6}
    print(rec)
    out.append(rec)
    eng.close()
json.dump(out, open(os.path.join(os.path.dirname(__file__), "..", "gpurun_out", "infer_sweep.json"), "w"), indent=1)
