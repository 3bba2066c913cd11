"""GELU / bias family vs swiglu / no-bias family at base size: egom2p_base_12e_12d_gelu against
egom2p_base_12e_12d_swiglu_nobias, the b = 32 dense training step (bench.py's flagship batch: 4 modalities, 2048 input +
2048 target tokens per sample, FusedAdamW with clip 1.0) and rgb -> depth guided generation (bench.py's rgb2depth
workload), the two models alternated step by step in one process so that both see the same clocks and neighbours.

The two MLPs have the same MACs per token (2 x 768 x 3072 = 3 x 768 x 2048), so the gap is the cost of the GELU family's
extra work: biases in the epilogues, the bias-gradient column sums and the LayerNorm bias gradients. Reports ms per step
(median and spread over the timed steps), nominal tokens/s, the per-family kernel split of one extra step under
ops.KernelTimer, generation latency, and the GPU's name, power limit and SM clock read in the same run.

    python tools/bench_model_family.py --steps 20 --warmup 3 --out profiles/family_b32.json
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

import bench  # noqa: E402  (batch layout and workloads of the flagship benchmark)

FAMILIES = ("egom2p_base_12e_12d_swiglu_nobias", "egom2p_base_12e_12d_gelu")


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         timeout=30).stdout.strip()
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {"error": "nvidia-smi gave no output"}


def build(name, dev):
    import egom2p_b200 as e
    from egom2p_b200.modality_info import MODALITY_INFO as MI
    torch.manual_seed(0)
    mods = e.MOD4
    m = e.create_model(name, encoder_embeddings={k: MI[k]["encoder_embedding"]() for k in mods},
                       decoder_embeddings={k: MI[k]["decoder_embedding"]() for k in mods},
                       modality_info={k: MI[k] for k in mods}, num_register_tokens=0)
    if name.endswith("_gelu"):   # non-zero biases, so that no epilogue can skip them
        with torch.no_grad():
            for n, p in m.named_parameters():
                if n.endswith(".bias"):
                    p.normal_(0.0, 0.02)
    return m.to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--gen-steps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_model_family.py measures on the GPU; no CUDA device found")
    from egom2p_b200 import ops
    from egom2p_b200.optim import FusedAdamW
    dev = torch.device("cuda", 0)
    B = args.batch
    md = {m: {k: v.to(dev) for k, v in d.items()} for m, d in bench.make_batch(B, 0, False).items()}
    models, opts = {}, {}
    for name in FAMILIES:
        models[name] = build(name, dev)
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
        for name in FAMILIES:
            step(name)
    info_start = gpu_info()
    ms = {name: [] for name in FAMILIES}
    for _ in range(args.steps):
        for name in FAMILIES:
            ms[name].append(timed(lambda: step(name)))
    info_end = gpu_info()
    split = {}
    for name in FAMILIES:
        with ops.KernelTimer() as kt:
            step(name)
        split[name] = {k: round(v["ms"], 3) for k, v in sorted(kt.summary().items(), key=lambda kv: -kv[1]["ms"])}

    # rgb -> depth guided generation (bench.py's rgb2depth workload: 5120 target tokens in 3 ROAR steps, CFG 2.0, batch 1)
    from egom2p_b200.generate import GenerationSampler, build_chained_generation_schedules, init_empty_target_modality, init_full_input_modality
    w = bench.GEN_WORKLOADS["rgb2depth"]
    schedule = build_chained_generation_schedules(
        cond_domains=[w["cond"]], target_domains=[w["target"]], tokens_per_target=[w["ntoks"]], autoregression_schemes=["roar"],
        decoding_steps=[w["steps"]], token_decoding_schedules=["linear"], temps=[0.01], temp_schedules=["constant"],
        cfg_scales=[2.0], cfg_schedules=["constant"], cfg_grow_conditioning=True)
    rng = np.random.default_rng(1234)
    tokens = torch.from_numpy(rng.integers(0, 64000, size=(w["batch"], 5, 32, 32), dtype=np.int64)).to(dev)
    gen_ms = {name: [] for name in FAMILIES}
    with torch.no_grad():
        samplers = {name: GenerationSampler(models[name].eval()) for name in FAMILIES}

        def gen(name):
            m = models[name]
            g = {w["cond"]: {"tensor": tokens}}
            g = init_empty_target_modality(g, m.modality_info, w["target"], w["batch"], w["ntoks"], dev)
            g = init_full_input_modality(g, m.modality_info, w["cond"], dev)
            samplers[name].generate(g, schedule, top_p=0.8, top_k=0.0, seed=0)
        for name in FAMILIES:
            gen(name)
        for _ in range(args.gen_steps):
            for name in FAMILIES:
                gen_ms[name].append(timed(lambda: gen(name)))

    tokens_per_step = B * bench.NOMINAL_TOKENS
    res = {"gpu": {"start": info_start, "end": info_end}, "batch": B, "steps": args.steps, "warmup": args.warmup,
           "regime": "dense, 2048 + 2048 tokens per sample, FusedAdamW + clip 1.0, fresh random init (seed 0)", "families": {}}
    for name in FAMILIES:
        a = np.array(ms[name])
        res["families"][name] = {
            "ms_per_step_median": float(np.median(a)), "ms_per_step_min": float(a.min()), "ms_per_step_max": float(a.max()),
            "ms_per_step_p10_p90": [float(np.percentile(a, 10)), float(np.percentile(a, 90))],
            "nominal_tokens_per_s": tokens_per_step / (float(np.median(a)) / 1e3),
            "kernel_ms_one_step": split[name],
            "rgb2depth_generation_ms": [round(x, 2) for x in gen_ms[name]]}
    g, s = (res["families"][n]["ms_per_step_median"] for n in reversed(FAMILIES))
    res["gelu_over_swiglu_step"] = g / s
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
