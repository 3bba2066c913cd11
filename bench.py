#!/usr/bin/env python
"""bench.py -- ego-b mod4 masked multimodal TRAINING step (BASELINE.json configs[1]) on N GPUs of one node.

A "step" = one pass of the hot path over one synthetic batch: H2D-free forward (index plan, fused embed/gather, 12
encoder + 12 decoder blocks, fused head + cross-entropy) + backward (+ DDP bucketed NCCL all-reduce for N > 1) +
clip_grad_norm_(1.0) + AdamW, exactly the body of the reference's train_one_epoch (run_training_egom2p.py:701-746).
Inputs: the "dense" synthetic regime of SURVEY.md section 8(d) (2048 encoder + 2048 decoder tokens per sample, all valid;
1009 rgb + 1009 depth + 15 cam + 15 gaze on both sides), random-init ego-b weights (396.2 M params), bf16 tensor-core
compute with fp32 masters / residual stream.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B_per_gpu] [--impl reference] [--dump-outputs DIR]

`value` = nominal tokens/s of the whole job (global batch x 4096 / step time, the reference's own accounting,
run_training_egom2p.py:645-647) timed on the device with inputs resident in HBM; `e2e` = the same metric through the
public model API with pinned-host inputs copied every step and the loss read back. `--impl reference` times the CPU
restatement of the reference path (oracle/, fp32, all host threads) on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy (float32): for training the loss, the
per-modality losses, the gradient norm and a fixed seeded sample of every parameter after the update; for generation the
generated tokens. Inputs, weights and the decoder modality order are seeded, so two builds run with the same arguments
can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NOMINAL_TOKENS = 4096  # num_input_tokens + num_target_tokens per sample
N_ENC = N_DEC = 2048
SPLIT = {"tok_rgb": 1009, "tok_depth": 1009, "tok_cam": 15, "tok_gaze": 15}
# algorithmic (mask-aware) FLOPs of one sample-step in the dense regime, SURVEY.md section 8(d): 3 x 1396.9 GFLOP
FLOP_PER_SAMPLE_STEP = 4190.6e9
# tokens per sample and vocabulary of each modality (egom2p/data/modality_info.py: tok_rgb / tok_depth = Cosmos DV4x8x8
# 5 x 32 x 32 tokens of a 64k codebook, tok_cam / tok_gaze = 30 tokens of a 256 codebook)
SHAPES = {"tok_cam": (30, 256), "tok_depth": (5120, 64000), "tok_gaze": (30, 256), "tok_rgb": (5120, 64000)}


def make_batch(b: int, seed: int, pin: bool):
    """Synthetic mod_dict in the reference layout (egom2p/data/masking.py:236-266), CPU tensors."""
    rng = np.random.default_rng(seed)
    md = {}
    for m in sorted(SHAPES):
        L, V = SHAPES[m]
        n = SPLIT[m]
        ids = rng.integers(0, V, size=(b, L), dtype=np.int64)
        imask = np.ones((b, L), dtype=bool)
        tmask = np.ones((b, L), dtype=bool)
        cnt = np.zeros((b, L), dtype=np.int32)
        for i in range(b):
            perm = rng.permutation(L)
            imask[i, perm[:n]] = False
            tmask[i, perm[n:2 * n]] = False
            cnt[i, int(np.argmin(tmask[i]))] = n
        t = torch.from_numpy(ids)
        if L == 5120:
            t = t.reshape(b, 5, 32, 32)
        d = {"tensor": t, "input_mask": torch.from_numpy(imask), "target_mask": torch.from_numpy(tmask),
             "decoder_attention_mask": torch.from_numpy(cnt)}
        md[m] = {k: (v.pin_memory() if pin else v) for k, v in d.items()}
    return md


def load_ref_masks():
    """Masks drawn by the reference's UnifiedMasking (oracle/gen_golden_masks.py): the ragged 'reference-distribution' regime."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_masks_egob.npz"))
    return g


def make_batch_ref_masks(b: int, offset: int, seed: int, pin: bool, g=None):
    g = load_ref_masks() if g is None else g
    rng = np.random.default_rng(seed)
    n = int(g["n"])
    sel = [(offset + i) % n for i in range(b)]
    md = {}
    for m in sorted(SHAPES):
        L, V = SHAPES[m]
        t = torch.from_numpy(rng.integers(0, V, size=(b, L), dtype=np.int64))
        if L == 5120:
            t = t.reshape(b, 5, 32, 32)
        imask = np.stack([np.unpackbits(g[m + "_input_mask"][i])[:L].astype(bool) for i in sel])
        tmask = np.stack([np.unpackbits(g[m + "_target_mask"][i])[:L].astype(bool) for i in sel])
        cnt = np.stack([g[m + "_attn"][i] for i in sel]).astype(np.int32)
        d = {"tensor": t, "input_mask": torch.from_numpy(imask), "target_mask": torch.from_numpy(tmask),
             "decoder_attention_mask": torch.from_numpy(cnt)}
        md[m] = {k: (v.pin_memory() if pin else v) for k, v in d.items()}
    return md


def step_flops(md) -> float:
    """Mask-aware algorithmic FLOPs of one training step on this batch (SURVEY.md section 8(d): 3 x forward)."""
    from egom2p_b200.modality_info import MODALITY_INFO as MI
    D, F, Le, Ld, N, M = 768, 2048, 12, 12, N_ENC, N_DEC
    mods = sorted(MI)
    b = md[mods[0]]["input_mask"].shape[0]
    total = 0.0
    for i in range(b):
        n_in = {m: int((~md[m]["input_mask"][i]).sum()) for m in mods}
        n_tg = {m: int((~md[m]["target_mask"][i]).sum()) for m in mods}
        n_enc = min(sum(n_in.values()), N)
        # targets are kept in modality order up to the budget
        left, kept = M, {}
        for m in mods:
            kept[m] = min(n_tg[m], left)
            left -= kept[m]
        n_dec = sum(kept.values())
        # valid tokens only: pad slots are don't-care rows (SURVEY A2) that the packed layout does not even compute
        enc = Le * (n_enc * (4 * D * D + 3 * D * F) + 2 * n_enc * n_enc * D)
        ctx = n_enc * D * D
        dec = Ld * (n_dec * (6 * D * D + 3 * D * F) + 2 * n_enc * D * D + 2 * sum(v * v for v in kept.values()) * D + 2 * n_dec * n_enc * D)
        head = sum(kept[m] * D * MI[m]["vocab_size"] for m in mods)
        total += 3 * 2.0 * (enc + ctx + dec + head)
    return total


def param_sample(model, k: int = 4096, seed: int = 0) -> dict:
    """A fixed, seeded sample of up to k elements of every parameter, as device tensors."""
    rng = np.random.default_rng(seed)
    out = {}
    for n, p in model.named_parameters():
        flat = p.detach().reshape(-1)
        idx = np.arange(flat.numel()) if flat.numel() <= k else np.sort(rng.choice(flat.numel(), k, replace=False))
        out[f"param.{n}"] = flat.index_select(0, torch.from_numpy(idx).to(flat.device))
    return out


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes every array as out_dir/<name>.npy in float32."""
    host = {n: np.asarray(a.detach().float().cpu() if torch.is_tensor(a) else a, dtype=np.float32) for n, a in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= 64 << 20, f"--dump-outputs: {total} bytes exceed the 64 MB budget"
    os.makedirs(out_dir, exist_ok=True)
    for n, a in host.items():
        np.save(os.path.join(out_dir, n + ".npy"), a)


def md_bytes(md):
    return int(sum(v.numel() * v.element_size() for d in md.values() for v in d.values()))


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with nvidia-smi while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower() == "active":
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=10)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def build_model(device):
    import egom2p_b200 as e
    from egom2p_b200.modality_info import MODALITY_INFO as MI
    torch.manual_seed(0)
    mods = e.MOD4
    model = e.create_model("egom2p_base_12e_12d_swiglu_nobias",
                           encoder_embeddings={k: MI[k]["encoder_embedding"]() for k in mods},
                           decoder_embeddings={k: MI[k]["decoder_embedding"]() for k in mods},
                           modality_info={k: MI[k] for k in mods}, num_register_tokens=0)
    # random-init ego-b weights: the deterministic draw the full-size parity fixtures were generated with (the reference's
    # init distributions, oracle/synth.make_state_dict seed 0), so the parity gate checks the very model that is timed
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gen_golden_egob as gg
    import synth
    model.load_state_dict(synth.make_state_dict(gg.egob_cfg(), gg.SD_SEED), strict=True)
    return model.to(device)


def parity_gate(model, dev):
    """The b = 1 full-size parity check of tests/test_egob_fullsize_gpu.py, run on the model that is about to be timed
    (SURVEY.md section 8(d): "parity gates run beside the timing"): loss / logits / gradient norms against the outputs of the
    UNMODIFIED reference in fp32 (tests/golden/egob_dense.npz, made by oracle/gen_golden_egob.py). oracle/ is used here as
    the checker only (deterministic weights + batch builders); nothing of it is timed."""
    import random
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gen_golden_egob as gg
    g = np.load(os.path.join(ROOT, "tests", "golden", "egob_dense.npz"))
    cfg = gg.egob_cfg()
    md = {m: {k: v.to(dev) for k, v in d.items()} for m, d in gg.dense_batch(cfg).items()}
    model.zero_grad(set_to_none=True)
    random.seed(gg.SHUFFLE_SEED)
    loss, mod_loss = model(md, N_ENC, N_DEC, loss_type="mod")
    loss.backward()
    ref = float(g["loss"])
    norms = dict(zip(g["grad_names"], g["grad_norms"]))
    gerr = max(abs(p.grad.double().norm().item() - norms[n]) / (norms[n] + 1e-12) for n, p in model.named_parameters())
    model.zero_grad(set_to_none=True)
    with torch.no_grad():
        random.seed(gg.SHUFFLE_SEED)
        logits = model(md, N_ENC, N_DEC, return_logits=True)
    cols = torch.from_numpy(g["cols"]).to(dev)
    lerr = {}
    for m in gg.MODS:
        rows = torch.from_numpy(g[f"rows::{m}"].astype(np.int64)).to(dev)
        lg = logits[m][0].index_select(0, rows).float()
        got = lg if lg.shape[-1] <= 256 else lg.index_select(1, cols)
        lerr[m] = float((got - torch.from_numpy(g[f"logits::{m}"]).to(dev)).abs().max())
    del logits
    out = {"case": "ego-b b=1 N=M=2048 dense split vs the unmodified reference in fp32 (tests/golden/egob_dense.npz)",
           "loss": float(loss), "loss_reference": ref, "loss_rel_err": abs(float(loss) - ref) / abs(ref),
           "logits_max_abs_err": lerr, "grad_norm_max_rel_err": gerr, "tolerances": {"loss_rel": 1e-3, "logits": 2e-2, "grad": 5e-2}}
    out["pass"] = bool(out["loss_rel_err"] < 1e-3 and max(lerr.values()) < 2e-2 and gerr < 5e-2)
    return out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


_CPU_REF = {}


def cpu_reference_step(b: int, threads: int):
    """One training step (fwd + bwd + clip_grad_norm_(1.0) + AdamW, the same body the GPU arm times) of the CPU fp32
    restatement (oracle/) on ego-b, dense regime, batch b, on `threads` host threads. Returns (seconds, loss). Weights and
    optimizer state persist across calls; building them is not timed."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import egom2p_oracle as orc
    import synth
    torch.set_num_threads(threads)
    if "leaf" not in _CPU_REF:
        cfg = synth.make_cfg(768, 12, 12, 12, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"])
        sd = synth.make_state_dict(cfg, 0)
        leaf = {}
        for k, v in sd.items():
            if k.endswith("to_logits.weight") or (k.startswith("decoder_embeddings") and k.endswith("mod_emb")):
                continue
            leaf[k] = v.requires_grad_(v.is_floating_point() and not k.endswith("pos_emb") and not (k.endswith(".bias") and "proj_context" not in k))
        train = {k: v for k, v in leaf.items() if v.requires_grad}
        opt = torch.optim.AdamW([{"params": [v for k, v in train.items() if not ("norm" in k or k.endswith(".bias"))], "weight_decay": 0.05},
                                 {"params": [v for k, v in train.items() if ("norm" in k or k.endswith(".bias"))], "weight_decay": 0.0}],
                                lr=1e-4, betas=(0.9, 0.95), eps=1e-8)
        for m in cfg["mods"]:
            leaf[f"decoder_embeddings.{m}.to_logits.weight"] = leaf[f"decoder_embeddings.{m}.token_emb.weight"]
            leaf[f"decoder_embeddings.{m}.mod_emb"] = leaf[f"encoder_embeddings.{m}.mod_emb"]
        _CPU_REF.update(cfg=cfg, leaf=leaf, train=list(train.values()), opt=opt, n=0)
    r = _CPU_REF
    md = make_batch(b, 1234 + r["n"], pin=False)
    r["n"] += 1
    t0 = time.perf_counter()
    out = orc.forward(r["leaf"], r["cfg"], md, N_ENC, N_DEC)
    out["loss"].backward()
    torch.nn.utils.clip_grad_norm_(r["train"], 1.0)
    r["opt"].step()
    r["opt"].zero_grad(set_to_none=True)
    return time.perf_counter() - t0, float(out["loss"])


def cpu_reference_arm(b: int, threads: int):
    """(seconds, loss, kind) of one CPU training step: the UNMODIFIED reference module (baseline/_ref, kind "reference") when
    tools/install_reference.py has put it there, else the oracle port (kind "port"). Same body either way: fp32 forward +
    backward + clip_grad_norm_(1.0) + AdamW on the dense synthetic batch, weights and optimizer state persistent."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import ref_gpu
    if not ref_gpu.available():
        return (*cpu_reference_step(b, threads), "port")
    torch.set_num_threads(threads)
    if "real" not in _CPU_REF:
        MI, create_model = ref_gpu.import_reference()
        mods = ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"]
        torch.manual_seed(0)
        model = create_model("egom2p_base_12e_12d_swiglu_nobias",
                             encoder_embeddings={m: MI[m]["encoder_embedding"]() for m in mods},
                             decoder_embeddings={m: MI[m]["decoder_embedding"]() for m in mods},
                             modality_info={m: MI[m] for m in mods}, num_register_tokens=0).train()
        decay = [p for n, p in model.named_parameters() if not ("norm" in n or n.endswith(".bias"))]
        no_decay = [p for n, p in model.named_parameters() if ("norm" in n or n.endswith(".bias"))]
        opt = torch.optim.AdamW([{"params": decay, "weight_decay": 0.05}, {"params": no_decay, "weight_decay": 0.0}],
                                lr=1e-4, betas=(0.9, 0.95), eps=1e-8)
        _CPU_REF["real"] = dict(model=model, opt=opt, params=list(model.parameters()), n=0)
    r = _CPU_REF["real"]
    md = {m: dict(d) for m, d in make_batch(b, 1234 + r["n"], pin=False).items()}
    r["n"] += 1
    t0 = time.perf_counter()
    loss, _ = r["model"](md, N_ENC, N_DEC, loss_type="mod")
    loss.backward()
    torch.nn.utils.clip_grad_norm_(r["params"], 1.0)
    r["opt"].step()
    r["opt"].zero_grad(set_to_none=True)
    return time.perf_counter() - t0, float(loss.detach()), "reference"


_KIND_TEXT = {"reference": "the unmodified reference module (baseline/_ref = /root/reference/egom2p), CPU fp32",
              "port": "oracle/egom2p_oracle.py (CPU fp32 restatement of the reference)"}


GEN_WORKLOADS = {  # eval_model_rgb2depth.py:45-59, eval_model_rgb2cam.py:40-54, eval_model_rgb2gaze.py:41-55, eval_model_depth2rgb.py:34-48
    "rgb2depth": dict(cond="tok_rgb", target="tok_depth", ntoks=5120, steps=3, batch=1, config=2),
    "rgb2cam": dict(cond="tok_rgb", target="tok_cam", ntoks=30, steps=3, batch=1, config=3),
    "rgb2gaze": dict(cond="tok_rgb", target="tok_gaze", ntoks=30, steps=5, batch=1, config=3),
    "depth2rgb": dict(cond="tok_depth", target="tok_rgb", ntoks=5120, steps=6, batch=64, config=4),
}


def generation_flops(w, schedule) -> float:
    """Algorithmic FLOPs of one clip through guided ROAR decoding in this repo's formulation (SURVEY.md section 8(d) formulas):
    per step a conditional and an unconditional encoder pass at their own lengths, one decoder pass per branch, ONE head."""
    D, F, Le, Ld = 768, 2048, 12, 12
    V = SHAPES[w["target"]][1]
    enc = lambda n: 2.0 * (Le * (n * (4 * D * D + 3 * D * F) + 2 * n * n * D) + n * D * D)
    dec = lambda k, n: 2.0 * Ld * (k * (6 * D * D + 3 * D * F) + 2 * n * D * D + 2 * k * k * D + 2 * k * n * D)
    done, total = 0, 0.0
    for st in schedule:
        k = int(st["num_tokens"])
        n_c, n_u = SHAPES[w["cond"]][0] + done, done
        total += enc(n_c) + enc(n_u) + dec(k, n_c) + dec(k, n_u) + 2.0 * k * D * V
        done += k
    return total


def run_generation(args):
    """BASELINE.json configs[2..4]: latency / throughput of guided ROAR generation through egom2p_b200.generate.GenerationSampler
    on synthetic conditioning tokens and random-init ego-b weights, with the unmodified reference sampler timed on the same GPU."""
    from egom2p_b200 import _lib
    from egom2p_b200.generate import GenerationSampler, build_chained_generation_schedules, init_empty_target_modality, init_full_input_modality
    w = GEN_WORKLOADS[args.workload]
    B = args.batch if args.batch_given else w["batch"]
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    model = build_model(dev).eval()
    info = model.modality_info
    sampler = GenerationSampler(model)
    schedule = build_chained_generation_schedules(
        cond_domains=[w["cond"]], target_domains=[w["target"]], tokens_per_target=[w["ntoks"]], autoregression_schemes=["roar"],
        decoding_steps=[w["steps"]], token_decoding_schedules=["linear"], temps=[0.01], temp_schedules=["constant"],
        cfg_scales=[2.0], cfg_schedules=["constant"], cfg_grow_conditioning=True)
    rng = np.random.default_rng(1234)
    n_calls = args.warmup + args.steps + 1
    host = [torch.from_numpy(rng.integers(0, 64000, size=(B, 5, 32, 32), dtype=np.int64)).pin_memory() for _ in range(n_calls)]
    devt = [t.to(dev) for t in host]

    def call(tokens):
        md = {w["cond"]: {"tensor": tokens}}
        md = init_empty_target_modality(md, info, w["target"], B, w["ntoks"], dev)
        md = init_full_input_modality(md, info, w["cond"], dev)
        return sampler.generate(md, schedule, top_p=0.8, top_k=0.0, seed=0)[w["target"]]["tensor"]

    def timed(fn, n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    with torch.no_grad():
        for i in range(args.warmup):
            call(devt[i])
        sampler_clk = ClockSampler(0)
        sampler_clk.start()
        l0 = _lib.launch_count()
        last = {}

        def timed_call(i):
            last["tokens"] = call(devt[args.warmup + i])
        ms = timed(timed_call, args.steps)
        launches = _lib.launch_count() - l0
        clocks = sampler_clk.stop()
        ms_e2e = timed(lambda i: call(host[args.warmup + i].to(dev, non_blocking=True)).cpu(), args.steps)
        # the same call as ONE CUDA graph (egom2p_b200.generate.GraphedGeneration): what is left when the ~1100 launches per
        # call are not issued from Python one at a time
        graph_ms = None
        if B <= 4:
            from egom2p_b200.generate import GraphedGeneration

            def mk(tokens):
                md = {w["cond"]: {"tensor": tokens}}
                md = init_empty_target_modality(md, info, w["target"], B, w["ntoks"], dev)
                return init_full_input_modality(md, info, w["cond"], dev)
            gg_ = GraphedGeneration(sampler, mk(devt[0]), schedule, top_p=0.8, top_k=0.0)
            mds = [mk(devt[args.warmup + i]) for i in range(args.steps)]
            for i in range(2):
                gg_(mds[i % len(mds)])
            graph_ms = timed(lambda i: gg_(mds[i]), args.steps) / args.steps
            del gg_
    t_call = ms / args.steps / 1e3
    flops = generation_flops(w, schedule) * B
    hbm, tf_burst, tf_sus, src = peaks()
    tfl = flops / t_call / 1e12
    line = {"metric": f"{args.workload} guided ROAR generation clips/sec", "value": B / t_call, "unit": "clips/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_call * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"BASELINE configs[{w['config']}]: {args.workload}, ego-b (396.2M) random-init, {SHAPES[w['cond']][0]} conditioning tokens -> "
                                   f"{w['ntoks']} target tokens in {w['steps']} ROAR steps, T = 0.01, top-p 0.8, CFG 2.0 (cond + uncond branch per step), "
                                   f"batch {B} clips per call; one step = one generate() call",
                       "batch": B, "latency_ms_per_clip_batch": t_call * 1e3, "latency_ms_cuda_graph": graph_ms,
                       "algorithmic_tflop_per_call": flops / 1e12,
                       "model_tflops": tfl, "mfu_vs_2250_spec": tfl / 2250.0, "mfu_vs_measured_sustained": tfl / tf_sus,
                       "l2_policy": "fresh conditioning tokens every call; activations exceed L2 for the video targets"},
            "e2e": {"value": B / (ms_e2e / args.steps / 1e3), "unit": "clips/s", "h2d_bytes_per_step": int(host[0].numel() * 8),
                    "d2h_bytes_per_step": int(B * w["ntoks"] * 8)},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "whole generate() call (GEMM + attention kernels)", "achieved": tfl, "peak": tf_sus,
                         "unit": "TFLOP/s", "frac": tfl / tf_sus, "traffic": None, "peak_source": f"{src} bf16_tflops_sustained"}}
    if not args.no_reference_gpu:
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import ref_gpu
        if ref_gpu.available():
            del sampler, model
            torch.cuda.empty_cache()
            res = []
            for rb in sorted({1, min(B, 4)}):
                try:
                    res.append(ref_gpu.time_reference_generation(args.workload, rb, 2, 1, dev))
                except torch.cuda.OutOfMemoryError:
                    res.append({"workload": args.workload, "batch": rb, "oom": True})
                    torch.cuda.empty_cache()
            line["reference_gpu"] = res
            best = max((r["clips_per_s"] for r in res if "clips_per_s" in r), default=None)
            if best:
                line["reference_gpu_speedup"] = line["value"] / best
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"tokens": last["tokens"]})
    print(json.dumps(line), flush=True)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    times = []
    kind = "port"
    for i in range(args.warmup + args.steps):
        dt, loss, kind = cpu_reference_arm(1, cores)
        if i >= args.warmup:
            times.append(dt)
    t = float(np.mean(times))
    val = NOMINAL_TOKENS / t
    line = {"impl": "reference", "metric": "ego-b mod4 train nominal tokens/sec (whole job)", "value": val, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "ego-b mod4 (396.2M) training step: fwd + bwd + clip_grad_norm(1.0) + AdamW, dense regime 2048 enc + 2048 dec "
                                   f"tokens/sample, CPU fp32, {_KIND_TEXT[kind]}, 1 sample per step",
                       "global_batch": 1},
            "cpu_baseline": {"value": val, "unit": "tokens/s", "cores": cores, "kind": kind,
                             "sample": f"1 sample (4096 nominal tokens) per step, fwd + bwd + clip + AdamW, {_KIND_TEXT[kind]}"},
            "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU (training: default 32; generation: the workload's batch)")
    ap.add_argument("--workload", default="train", choices=["train"] + list(GEN_WORKLOADS),
                    help="train: the ego-b mod4 training step (the headline, BASELINE configs[1]); others: guided ROAR generation (configs[2..4])")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--regime", default="dense", choices=["dense", "reference-masks"],
                    help="dense: SURVEY 8(d) headline synthetic regime; reference-masks: ragged masks drawn by the reference's UnifiedMasking")
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"],
                    help="fused: egom2p_b200.optim.FusedAdamW (multi-tensor clip + AdamW); torch: clip_grad_norm_ + torch.optim.AdamW(fused=True)")
    ap.add_argument("--allreduce", default="fp32", choices=["fp32", "bf16"],
                    help="gradient all-reduce precision for N > 1 (fp32 = the reference's DDP default; bf16 = torch's bf16_compress_hook)")
    ap.add_argument("--bucket-mb", type=int, default=100,
                    help="DDP gradient bucket size (MB) for N > 1: 16 all-reduce launches per step instead of 64 at torch's default 25 MB "
                         "(each NCCL kernel that co-runs with the backward takes SM pairs from the GEMMs; same box, N = 2: 195.1 / 193.0 / 192.5 ms "
                         "at 25 / 100 / 400 MB against 184.9 ms on one GPU)")
    ap.add_argument("--no-batch4", action="store_true", help="skip the extra b = 4 per GPU measurement (the reference's own batch size; N = 1 only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the b = 1 full-size parity gate against the reference's fp32 outputs")
    ap.add_argument("--no-reference-gpu", action="store_true",
                    help="skip timing the unmodified reference (baseline/_ref, eager bf16 autocast) on this GPU (N = 1 only)")
    ap.add_argument("--cpu-steps", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU paths (--impl ours)")
    args.batch_given = args.batch is not None
    if args.batch is None:
        args.batch = int(os.environ.get("EGOM2P_BENCH_BATCH", "32"))
    if args.workload != "train":
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the CPU reference arm times the training step only (--workload train)"}))
            return
        args.warmup = max(args.warmup, 1) if args.workload == "depth2rgb" else max(args.warmup, 3)
        return run_generation(args)
    if args.impl == "reference":
        args.warmup = min(args.warmup, 1)
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    from egom2p_b200 import _lib, ops
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # The GEMM runs as CTA pairs that need both SMs of a TPC, so every SM an NCCL channel occupies during the overlapped
        # gradient all-reduce takes a whole pair away from it; 16 channels saturate NVLink 5 for this message size
        # (8 GPUs: 205.0 ms / step against 207.3 with NCCL's default channel count).
        os.environ.setdefault("NCCL_MAX_CTAS", "16")
        dist.init_process_group("nccl", device_id=dev)
    b = args.batch
    model = build_model(dev)
    net = model
    if world > 1:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=False,
                                                        broadcast_buffers=False, gradient_as_bucket_view=True,
                                                        bucket_cap_mb=args.bucket_mb)
        if args.allreduce == "bf16":   # optional gradient compression: halves the NVLink bytes of the overlapped all-reduce
            from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
            net.register_comm_hook(None, default_hooks.bf16_compress_hook)
    decay = [p for n, p in model.named_parameters() if not ("norm" in n or n.endswith(".bias"))]
    no_decay = [p for n, p in model.named_parameters() if ("norm" in n or n.endswith(".bias"))]
    groups = [{"params": decay, "weight_decay": 0.05}, {"params": no_decay, "weight_decay": 0.0}]
    if args.optimizer == "fused":   # the device-side tail of this repo: grad-norm + AdamW in two launches over all 245 tensors
        from egom2p_b200.optim import FusedAdamW
        opt = FusedAdamW(groups, lr=1e-4, betas=(0.9, 0.95), eps=1e-8)
    else:
        opt = torch.optim.AdamW(groups, lr=1e-4, betas=(0.9, 0.95), eps=1e-8, fused=True)
    params = list(model.parameters())

    # a fresh batch for every warm-up and timed step (seed = 1234 + rank * 1000 + step, SURVEY.md section 8(d)): nothing to memorise
    nb = args.warmup + args.steps
    if args.regime == "dense":
        host_batches = [make_batch(b, 1234 + rank * 1000 + s, pin=True) for s in range(nb)]
        flops_per_step = b * FLOP_PER_SAMPLE_STEP
    else:
        gm = load_ref_masks()
        host_batches = [make_batch_ref_masks(b, (rank * nb + s) * b, 1234 + rank * 1000 + s, pin=True, g=gm) for s in range(nb)]
        flops_per_step = float(np.mean([step_flops(hb) for hb in host_batches[args.warmup:]]))
    dev_batches = [{m: {k: v.to(dev) for k, v in d.items()} for m, d in hb.items()} for hb in host_batches]

    def step(md):
        loss, mod_loss = net(md, N_ENC, N_DEC, loss_type="mod")
        loss.backward()
        if args.optimizer == "fused":
            grad_norm = opt.clip_grad_norm_(1.0)
        else:
            grad_norm = torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss, mod_loss, grad_norm

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        sync()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- parity gate on the model about to be timed (b = 1, full size, against the unmodified reference's fp32 outputs)
    parity = None
    if not args.no_parity:
        try:
            parity = parity_gate(model, dev)
        except Exception as exc:  # noqa: BLE001  (reported in the line; the timing still runs)
            parity = {"pass": False, "error": f"{type(exc).__name__}: {exc}"[:300]}
            model.zero_grad(set_to_none=True)

    # ---- warm-up, then device-resident timing
    random.seed(0)   # the decoder modality order, so that every run computes the same steps
    for i in range(args.warmup):
        step(dev_batches[i])
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = _lib.launch_count()
    last = {}

    def timed_step(i):
        last["out"] = step(dev_batches[args.warmup + i])
    ms = timed(timed_step, args.steps)
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    outputs = None
    if args.dump_outputs and rank == 0:   # before the steps below move the weights on
        loss, mod_loss, grad_norm = last["out"]
        outputs = {"loss": loss, "grad_norm": grad_norm, **{f"mod_loss.{m}": v for m, v in mod_loss.items()},
                   **param_sample(model)}

    # ---- end-to-end through the public API: pinned host inputs copied every step, loss read back every step
    def e2e_step(i):
        md = {m: {k: v.to(dev, non_blocking=True) for k, v in d.items()} for m, d in host_batches[args.warmup + i].items()}
        return step(md)[0].item()
    e2e_step(0)
    ms_e2e = timed(e2e_step, args.steps)
    last_loss = e2e_step(0)

    # ---- the reference's own per-GPU batch (4): eager, and as one CUDA graph per step (egom2p_b200/graphed.py)
    batch4 = None
    if world == 1 and not args.no_batch4 and args.regime == "dense" and args.optimizer == "fused":
        try:   # auxiliary measurement: a failure here must not cost the headline line
            from egom2p_b200.graphed import GraphedTrainStep
            from egom2p_b200.optim import FusedAdamW
            nb4 = args.steps * 2
            b4 = [{m: {k: v.to(dev) for k, v in d.items()} for m, d in make_batch(4, 777 + s, pin=False).items()} for s in range(nb4 + 1)]
            for i in range(3):
                step(b4[i])
            l0 = _lib.launch_count()
            ms4 = timed(lambda i: step(b4[i]), nb4)
            l4 = (_lib.launch_count() - l0) / nb4
            opt.zero_grad(set_to_none=True)
            opt4 = FusedAdamW(groups, lr=1e-4, betas=(0.9, 0.95), eps=1e-8)
            runner = GraphedTrainStep(model, opt4, b4[nb4], N_ENC, N_DEC, clip_grad=1.0)
            for i in range(3):
                runner(b4[i])
            ms4g = timed(lambda i: runner(b4[i]), nb4)
            model.static_target_rows = None
            model.fixed_decoder_order = None
            del runner, opt4
            mk4 = lambda ms_: {"ms_per_step": ms_ / nb4, "tokens_per_s": 4 * NOMINAL_TOKENS / (ms_ / nb4 / 1e3),
                               "mfu_vs_2250_spec": 4 * FLOP_PER_SAMPLE_STEP / (ms_ / nb4 / 1e3) / 1e12 / 2250.0}
            batch4 = {"what": "same training step at b = 4 per GPU (the reference's batch_size), dense regime, steps = %d" % nb4,
                      "eager": dict(mk4(ms4), launches_per_step=l4),
                      "cuda_graph": dict(mk4(ms4g), launches_per_step=1, note="whole step (fwd + bwd + clip + AdamW) replayed as one graph")}
        except Exception as exc:  # noqa: BLE001
            model.static_target_rows = None
            model.fixed_decoder_order = None
            batch4 = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- data-parallel consistency: after the timed steps every rank must hold the same weights (same all-reduced gradients,
    # same optimizer arithmetic); checked on a checksum of all parameters
    ddp_check = None
    if world > 1:
        chk = torch.stack([torch.stack([p.detach().double().sum(), p.detach().double().abs().sum()]) for p in model.parameters()]).sum(0)
        allc = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        allc = torch.stack(allc)
        ddp_check = {"ranks": world, "weights_identical_across_ranks": bool((allc == allc[0]).all()),
                     "checksum": [float(v) for v in allc[0]], "allreduce": args.allreduce}

    # ---- per-kernel-family breakdown of one extra step (CUDA events around each C-ABI launch)
    with ops.KernelTimer() as kt:
        step(dev_batches[0])
    fam = kt.summary()

    if rank == 0:
        t_step = ms / args.steps / 1e3
        gbatch = b * world
        value = gbatch * NOMINAL_TOKENS / t_step
        e2e_val = gbatch * NOMINAL_TOKENS / (ms_e2e / args.steps / 1e3)
        hbm, tf_burst, tf_sus, src = peaks()
        tflops = flops_per_step / t_step / 1e12  # per GPU (rank 0's batches; mask-aware FLOPs in the ragged regime)
        g = fam.get("gemm", {"ms": 1e-9, "work": 0.0, "launches": 1})
        achieved = g["work"] / (g["ms"] / 1e3) / 1e12
        total_kernel_ms = sum(d["ms"] for d in fam.values())
        line = {
            "metric": "ego-b mod4 train nominal tokens/sec (whole job)", "value": value, "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "ego-b mod4 (egom2p_base_12e_12d_swiglu_nobias, 396.2M params) training step: fwd + bwd + "
                                   "clip_grad_norm(1.0) + AdamW; " +
                                   ("dense synthetic regime, 2048 encoder + 2048 decoder tokens/sample "
                                    "(1009 rgb + 1009 depth + 15 cam + 15 gaze per side)" if args.regime == "dense" else
                                    "reference-distribution regime: masks drawn by the reference UnifiedMasking (budgets 2048 / 2048, "
                                    "ragged: mean 1086 valid inputs / 891 valid targets), mask-aware FLOPs") + ", random-init weights",
                       "regime": args.regime,
                       "global_batch": gbatch, "batch_per_gpu": b, "parallelism": f"dp{world}", "nominal_tokens_per_sample": NOMINAL_TOKENS,
                       "l2_policy": "working set (activations + 1.6 GB weights) far exceeds the 126 MB L2; no explicit flush",
                       "model_tflops_per_gpu": tflops, "mfu_vs_2250_spec": tflops / 2250.0,
                       "mfu_vs_measured_sustained": tflops / tf_sus, "peaks_source": src, "loss": last_loss},
            "e2e": {"value": e2e_val, "unit": "tokens/s", "h2d_bytes_per_step": md_bytes(host_batches[0]), "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches),
            "parity": parity,
            "batch4": batch4,
            "ddp": ddp_check,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "gemm_kernel (tcgen05 bf16 GEMM, all nn.Linear fwd/dgrad/wgrad)",
                         "achieved": achieved, "peak": tf_sus, "unit": "TFLOP/s", "frac": achieved / tf_sus,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of the qkv projection
                         # launch of this workload (b = 32: M = 65536, N = 2304, K = 768; algorithmic bytes 406 MB): profiles/r01e_gemm_ncu.md
                         "traffic": 354.5e6, "traffic_unit": "bytes per launch (M=65536 N=2304 K=768 projection, b=32)",
                         "peak_source": f"{src} bf16_tflops_sustained (kernel timed inside a long step)",
                         "share_of_kernel_time": g["ms"] / max(total_kernel_ms, 1e-9),
                         "families": {k: {"ms": round(d["ms"], 3), "launches": d["launches"],
                                          ("tflops" if d["unit"] == "flop" else "gbs"):
                                              round(d["work"] / (d["ms"] / 1e3 + 1e-12) / (1e12 if d["unit"] == "flop" else 1e9), 1)}
                                      for k, d in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}},
        }
        if world == 1 and not args.no_cpu_baseline:   # rank 0 at N = 1 only
            cores = os.cpu_count() or 1
            try:
                res = [cpu_reference_arm(1, cores) for _ in range(args.cpu_steps)]
                dt, kind = float(np.mean([r[0] for r in res])), res[-1][2]
            except Exception as exc:  # noqa: BLE001  (auxiliary measurement)
                dt, kind = float("nan"), "port"
                line["cpu_baseline_error"] = f"{type(exc).__name__}: {exc}"[:300]
            line["cpu_baseline"] = {"value": NOMINAL_TOKENS / dt, "unit": "tokens/s", "cores": cores, "kind": kind,
                                    "sample": f"{args.cpu_steps} x (1 sample = 4096 nominal tokens, fwd + bwd + clip + AdamW, fp32) of the same dense workload, {_KIND_TEXT[kind]}"}
        if world == 1 and not args.no_reference_gpu:
            # the bar to beat: the unmodified reference on this same GPU (baseline/ref_gpu.py); our model is released first
            sys.path.insert(0, os.path.join(ROOT, "baseline"))
            import ref_gpu
            if ref_gpu.available():
                del opt, params, net, model, dev_batches, groups, decay, no_decay
                import gc
                gc.collect()
                torch.cuda.empty_cache()
                res = []
                for rb in (4, 8):
                    try:
                        res.append(ref_gpu.time_reference(rb, 20, 5, dev, make_batch))
                    except torch.cuda.OutOfMemoryError:
                        res.append({"batch_per_gpu": rb, "oom": True})
                        torch.cuda.empty_cache()
                    except Exception as exc:  # noqa: BLE001  (auxiliary measurement)
                        res.append({"batch_per_gpu": rb, "error": f"{type(exc).__name__}: {exc}"[:300]})
                        torch.cuda.empty_cache()
                line["reference_gpu"] = res
                best = max((r["tokens_per_s"] for r in res if "tokens_per_s" in r), default=None)
                if best:
                    line["reference_gpu_speedup"] = value / best
            else:
                line["reference_gpu"] = {"unavailable": "baseline/_ref/egom2p missing (tools/install_reference.py)"}
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
