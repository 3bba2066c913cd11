"""TEST INFRASTRUCTURE ONLY. Runs the UNMODIFIED reference GenerationSampler (egom2p/models/generate.py, imported from
/root/reference in the authoring container) on a small 4-modality model and records every call it makes into the model
(forward_encoder / decoder_proj_context / forward_decoder / forward_logits: inputs and outputs) for

  * rgb -> cam   (BASELINE.json configs[3]: eval_model_rgb2cam.py:40-59 -- ROAR, 3 steps, cfg 2.0, temperature 0.01, top-p 0.8)
  * rgb -> depth (configs[2]: eval_model_rgb2depth.py -- ROAR over the video tokens, same guidance settings)

Sampling itself is random (torch.multinomial); the recorded calls are what pins the model side of the sampler surface
(SURVEY.md section 8, row a22): tests/test_sampler_surface_gpu.py replays each call's inputs through the B200 module.
Run: `python oracle/gen_golden_sampler.py`  -> tests/golden/sampler_calls_small4_{tok_cam,tok_depth}.npz (one file per run,
packed by `pack` to stay under 1 MB each)
"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import synth  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def pack(store):
    """Shrinks one run's recorded calls without changing what the replay test checks. An array equal to one stored earlier
    in the same run is stored once; the later key holds the 0-d string "@<earlier key>". An expected value that is no call's
    input (an encoder output, logits) is stored in float16 with "<key>_qerr", the largest |float32 - float16| over it: the
    replay subtracts it from its tolerance, so passing against the float16 values implies passing against the float32 ones."""
    out, seen = {}, {}
    for k, a in store.items():
        if a.dtype == np.float32 and ((k.endswith("_out") and "forward_encoder" in str(store[k[:4] + "_name"])) or "_logits_" in k):
            a16 = a.astype(np.float16)
            out[k], out[k + "_qerr"] = a16, np.float32(np.abs(a16.astype(np.float32) - a).max() if a.size else 0.0)
            continue
        h = hashlib.sha1(a.dtype.str.encode() + str(a.shape).encode() + a.tobytes()).hexdigest()
        if a.dtype.kind in "fiub" and a.nbytes > 64 and h in seen:
            out[k] = np.array("@" + seen[h])
        else:
            seen.setdefault(h, k)
            out[k] = a
    return out


class Packed:
    """Reads a file written by `pack`: resolves "@<key>" back-references and returns, with each
    expected value, its tolerance less the float16 rounding bound stored beside it."""

    def __init__(self, path):
        self.g = np.load(path)

    def __contains__(self, k):
        return k in self.g.files

    def __getitem__(self, k):
        a = self.g[k]
        if a.ndim == 0 and a.dtype.kind == "U" and str(a).startswith("@"):
            a = self.g[str(a)[1:]]
        return a

    def expected(self, k, tol):
        q = float(self.g[k + "_qerr"]) if k + "_qerr" in self else 0.0
        return self[k].astype(np.float32), tol - q


def main():
    from gen_golden import build_ref  # imports the reference
    from egom2p.models.generate import (GenerationSampler, build_chained_generation_schedules, init_empty_target_modality,
                                        init_full_input_modality)
    torch.manual_seed(0)
    cfg = synth.make_cfg(192, 3, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=512, video_thw=(5, 4, 4))
    model = build_ref(cfg).eval()
    model.load_state_dict(synth.make_state_dict(cfg, 17), strict=True)
    info = model.modality_info
    calls = []

    def to_np(t):
        if t is None:
            return None
        return t.detach().cpu().numpy()

    def record(name, fn):
        def wrapped(*a, **kw):
            out = fn(*a, **kw)
            calls.append((name, a, kw, out))
            return out
        return wrapped

    model.forward_encoder = record("forward_encoder", model.forward_encoder)
    model.forward_decoder = record("forward_decoder", model.forward_decoder)
    model.forward_logits = record("forward_logits", model.forward_logits)
    sampler = GenerationSampler(model)
    gen = torch.Generator().manual_seed(5)
    L = cfg["mods"]["tok_rgb"]["len"]
    rgb = torch.randint(0, 512, (1, 5, 4, 4), generator=gen)
    for target, ntok, steps in (("tok_cam", 30, 3), ("tok_depth", L, 3)):
        schedule = build_chained_generation_schedules(
            cond_domains=["tok_rgb"], target_domains=[target], tokens_per_target=[ntok], autoregression_schemes=["roar"],
            decoding_steps=[steps], token_decoding_schedules=["linear"], temps=[0.01], temp_schedules=["constant"],
            cfg_scales=[2.0], cfg_schedules=["constant"], cfg_grow_conditioning=True)
        sample = {"tok_rgb": {"tensor": rgb.clone(), "input_mask": torch.zeros(1, L, dtype=torch.bool),
                              "target_mask": torch.ones(1, L, dtype=torch.bool)}}
        sample = init_empty_target_modality(sample, info, target, 1, ntok, "cpu")
        sample = init_full_input_modality(sample, info, "tok_rgb", "cpu")
        calls.clear()
        store, n = {}, 0
        with torch.no_grad():
            sampler.generate(sample, schedule, verbose=False, seed=0, top_p=0.8, top_k=0.0)
        for name, a, kw, out in calls:
            pre = f"c{n:03d}"
            store[pre + "_name"] = np.array(f"{target}:{name}")
            if name == "forward_encoder":
                store[pre + "_x"], store[pre + "_mask"], store[pre + "_out"] = to_np(a[0]), to_np(kw.get("encoder_mask", a[1] if len(a) > 1 else None)), to_np(out)
            elif name == "forward_decoder":
                y, ctx, emask, dmask = (list(a) + [None] * 4)[:4]
                emask = kw.get("encoder_mask", emask)
                dmask = kw.get("decoder_attention_mask", dmask)
                store[pre + "_y"], store[pre + "_ctx"], store[pre + "_emask"] = to_np(y), to_np(ctx), to_np(emask)
                if dmask is not None:
                    store[pre + "_dmask"] = to_np(dmask)
                store[pre + "_out"] = to_np(out)
            else:  # forward_logits(y, decoder_mod_dict, decoder_mod_mask[, return_all_logits])
                y, dmd, dmm = a[0], a[1], a[2]
                store[pre + "_y"], store[pre + "_modmask"] = to_np(y), to_np(dmm)
                store[pre + "_mods"] = np.array(list(dmd.keys()))
                store[pre + "_all"] = np.array(bool(kw.get("return_all_logits", a[3] if len(a) > 3 else False)))
                for m, lg in out.items():
                    store[pre + "_logits_" + m] = to_np(lg)
            n += 1
        store["n_calls"] = np.array(n)
        store["sd_seed"] = np.array(17)
        np.savez_compressed(os.path.join(OUT, f"sampler_calls_small4_{target}.npz"), **pack(store))
        names = [str(store[f"c{i:03d}_name"]) for i in range(n)]
        print(n, "calls:", names)
        for i in range(n):
            pre = f"c{i:03d}"
            print(" ", names[i], {k[len(pre) + 1:]: store[k].shape for k in store if k.startswith(pre) and k != pre + "_name" and hasattr(store[k], "shape")})


if __name__ == "__main__":
    main()
