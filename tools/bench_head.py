"""The vocabulary head alone: decoder_norm -> one 64k-vocabulary head -> cross-entropy, forward + backward
(egom2p_b200.model._HeadLossFn) at the row count of one 64k modality of the flagship step (ego-b, b = 32 dense: R = 32 288
target rows, V = 64 000, D = 768), with a random-init table (std 0.02, as the model initialises it).

Reports the median and spread of forward + backward over the timed iterations (CUDA events, each iteration ends in a
synchronise), the per-family kernel split of one extra iteration under ops.KernelTimer, the cost of the loss pass's
fall-back launch when no 128-row tile is flagged (what every step pays when all rows are exact) next to a small
elementwise launch, the loss pass with and without storing the softmax numerators (device times from CUDA-graph replays),
and the GPU's name, power limit and SM clock read in the same run.

    python tools/bench_head.py --iters 20 --warmup 3
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         timeout=30).stdout.strip()
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {"error": "nvidia-smi gave no output"}


def graph_us(fn, launches=100):
    """Device time of one fn() call: `launches` calls captured as one CUDA graph and replayed (no host launch cost)."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(launches):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return 1000.0 * e0.elapsed_time(e1) / launches


def loss_pass_costs(ops, y, w, tgt):
    """Device times (us) of the loss pass with and without storing the numerators, of the gated fall-back launch when no
    tile is flagged, and, for scale, of a small elementwise launch (the backward's row scaling)."""
    R, V = y.shape[0], w.shape[0]
    _, lse, (probs, rscale, _) = ops.ce_forward(y, w, tgt, keep_probs=True)
    flags = torch.zeros((R + 127) // 128, dtype=torch.uint8, device=y.device)
    gscale = torch.ones(1, device=y.device)
    return {"loss_pass_stats_only_us": graph_us(lambda: ops.ce_forward(y, w, tgt), 10),
            "loss_pass_storing_probs_us": graph_us(lambda: ops.ce_forward(y, w, tgt, keep_probs=True), 10),
            "empty_fallback_launch_us": graph_us(lambda: ops.ce_dlogits(y, w, tgt, lse, None, 0, V, probs, tile_flag=flags)),
            "row_scale_launch_us": graph_us(lambda: ops.ce_row_scale(y, rscale, gscale, want_ys=False))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=32288)
    ap.add_argument("--vocab", type=int, default=64000)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_head.py measures on the GPU; no CUDA device found")
    from egom2p_b200 import model as M
    from egom2p_b200 import ops
    dev = torch.device("cuda", 0)
    D, R, V = 768, args.rows, args.vocab
    g = torch.Generator(device=dev).manual_seed(0)
    S = 2 * R   # decoder rows of which the head takes R (the other modality's rows get a zero gradient)
    y = torch.randn(S, D, generator=g, device=dev)
    idx = torch.randperm(S, generator=g, device=dev)[:R].sort().values
    tgt = torch.randint(0, V, (R,), generator=g, device=dev)
    w = torch.nn.Parameter(torch.randn(V, D, generator=g, device=dev) * 0.02)
    wb = w.detach().bfloat16()
    yd = y.requires_grad_(True)
    nw = torch.nn.Parameter(torch.ones(D, device=dev))

    def step():
        yd.grad = nw.grad = w.grad = None
        loss = M._HeadLossFn.apply(yd, nw, None, [idx], [tgt], [wb], 1e-6, [0], True, w)[0]
        loss.backward()

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for _ in range(args.warmup):
        step()
    info_start = gpu_info()
    ms = np.array([timed(step) for _ in range(args.iters)])
    info_end = gpu_info()
    with ops.KernelTimer() as kt:
        step()
    split = {k: {"ms": round(v["ms"], 3), "launches": v["launches"]}
             for k, v in sorted(kt.summary().items(), key=lambda kv: -kv[1]["ms"])}
    ym = ops.layernorm_fwd(y.detach(), nw.detach(), 1e-6)[0].index_select(0, idx)
    res = {"gpu": {"start": info_start, "end": info_end}, "rows": R, "vocab": V, "dim": D, "iters": args.iters,
           "warmup": args.warmup, "ms_fwd_bwd_median": float(np.median(ms)), "ms_fwd_bwd_min": float(ms.min()),
           "ms_fwd_bwd_max": float(ms.max()), "head_flop_per_pass": 2.0 * R * V * D, "kernel_ms_one_iter": split,
           **loss_pass_costs(ops, ym, wb, tgt)}
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
