"""Cost of a training step with frozen parameters: the ego-b b = 32 dense step (bench.py's flagship batch: 4 modalities,
2048 input + 2048 target tokens per sample, FusedAdamW with clip 1.0) with nothing frozen, under freeze_shared_params()
(encoder and decoder blocks and norms frozen; embeddings, heads and the context projection train) and under
freeze_encoder(freeze_embeddings=True) (decoder-side training). One model per configuration, all three built from the same
weights and stepped in turn, so that they see the same clocks and neighbours. The autograd nodes skip the gradient work of
frozen parameters (weight-gradient GEMMs, bias and LayerNorm reductions, head dW, frozen embedding tables), so the frozen
steps should be cheaper; the unfrozen step is the flagship step itself.

Reports ms per step (median and spread over the timed steps), the per-family kernel split of one extra step under
ops.KernelTimer, and the GPU's name, power limit and SM clock read in the same run.

    python tools/bench_frozen.py --steps 20 --warmup 3 --out profiles/frozen_b32.json
"""
import argparse
import json
import os
import random
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (batch layout and model of the flagship benchmark)

CONFIGS = {
    "none": lambda m: None,
    "freeze_shared_params": lambda m: m.freeze_shared_params(),
    "freeze_encoder": lambda m: m.freeze_encoder(freeze_embeddings=True),
}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         timeout=30).stdout.strip()
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {"error": "nvidia-smi gave no output"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_frozen.py measures on the GPU; no CUDA device found")
    from egom2p_b200 import ops
    from egom2p_b200.optim import FusedAdamW
    dev = torch.device("cuda", 0)
    B = args.batch
    md = {m: {k: v.to(dev) for k, v in d.items()} for m, d in bench.make_batch(B, 0, False).items()}
    models, opts = {}, {}
    for name, freeze in CONFIGS.items():
        models[name] = bench.build_model(dev)
        freeze(models[name])
        opts[name] = FusedAdamW([{"params": [p for p in models[name].parameters() if p.requires_grad], "weight_decay": 0.05}],
                                lr=1e-4, betas=(0.9, 0.95))

    def step(name):
        model, opt = models[name], opts[name]
        loss, _ = model(md, bench.N_ENC, bench.N_DEC)
        loss.backward()
        opt.clip_grad_norm_(1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    random.seed(0)
    for _ in range(args.warmup):
        for name in CONFIGS:
            step(name)
    info_start = gpu_info()
    ms = {name: [] for name in CONFIGS}
    for _ in range(args.steps):
        for name in CONFIGS:
            ms[name].append(timed(lambda: step(name)))
    info_end = gpu_info()
    split = {}
    for name in CONFIGS:
        with ops.KernelTimer() as kt:
            step(name)
        split[name] = {k: round(v["ms"], 3) for k, v in sorted(kt.summary().items(), key=lambda kv: -kv[1]["ms"])}

    res = {"gpu": {"start": info_start, "end": info_end}, "batch": B, "steps": args.steps, "warmup": args.warmup,
           "regime": "ego-b (egom2p_base_12e_12d_swiglu_nobias), dense, 2048 + 2048 tokens per sample, FusedAdamW + clip 1.0",
           "configs": {}}
    for name in CONFIGS:
        a = np.array(ms[name])
        res["configs"][name] = {
            "ms_per_step_median": float(np.median(a)), "ms_per_step_min": float(a.min()), "ms_per_step_max": float(a.max()),
            "ms_per_step_p10_p90": [float(np.percentile(a, 10)), float(np.percentile(a, 90))],
            "trainable_params": sum(p.numel() for p in models[name].parameters() if p.requires_grad),
            "kernel_ms_one_step": split[name]}
    base = res["configs"]["none"]["ms_per_step_median"]
    res["step_over_unfrozen"] = {name: res["configs"][name]["ms_per_step_median"] / base for name in CONFIGS}
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
