"""GPU: the model side of the generation sampler (SURVEY.md section 8 row a22; BASELINE.json configs[2] rgb -> depth and
configs[3] rgb -> cam). tests/golden/sampler_calls_small4_{tok_cam,tok_depth}.npz hold every call the UNMODIFIED reference
GenerationSampler made into its model during guided ROAR decoding (oracle/gen_golden_sampler.py: forward_encoder /
forward_decoder / forward_logits, conditional and unconditional passes, context lengths 0 .. 134, no decoder mask). Each call's
inputs are replayed through the B200 module holding the same weights. Tolerances: logits 2e-2 max-abs (BASELINE.json
north_star); encoder / decoder activations 3e-2 max-abs on O(1) LayerNorm outputs (bf16 tensor-core compute vs the fp32
reference), less the rounding bound of the expected values stored in float16 (oracle/gen_golden_sampler.pack)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import synth  # noqa: E402
from gen_golden_sampler import Packed  # noqa: E402
from test_model_gpu import build_model  # noqa: E402


def test_reference_sampler_calls_replayed(golden_dir):
    cfg = synth.make_cfg(192, 3, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=512, video_thw=(5, 4, 4))
    model = build_model(cfg).cuda().eval()
    cu = lambda a: torch.from_numpy(np.asarray(a)).cuda()
    seen = set()
    for target in ("tok_cam", "tok_depth"):
        g = Packed(os.path.join(golden_dir, f"sampler_calls_small4_{target}.npz"))
        model.load_state_dict(synth.make_state_dict(cfg, int(g["sd_seed"])), strict=True)
        with torch.no_grad():
            for i in range(int(g["n_calls"])):
                pre = f"c{i:03d}"
                t, name = str(g[pre + "_name"]).split(":")
                assert t == target
                seen.add(name)
                if name == "forward_encoder":
                    out = model.forward_encoder(cu(g[pre + "_x"]), encoder_mask=cu(g[pre + "_mask"]))
                    ref, tol = g.expected(pre + "_out", 3e-2)
                    assert tuple(out.shape) == ref.shape
                    if ref.size:
                        assert float((out.float().cpu() - torch.from_numpy(ref)).abs().max()) < tol, (target, i, name)
                elif name == "forward_decoder":
                    dmask = cu(g[pre + "_dmask"]) if pre + "_dmask" in g else None
                    out = model.forward_decoder(cu(g[pre + "_y"]), cu(g[pre + "_ctx"]), encoder_mask=cu(g[pre + "_emask"]),
                                                decoder_attention_mask=dmask)
                    ref, tol = g.expected(pre + "_out", 3e-2)
                    assert tuple(out.shape) == ref.shape
                    assert float((out.float().cpu() - torch.from_numpy(ref)).abs().max()) < tol, (target, i, name, ref.shape, g[pre + "_ctx"].shape)
                else:
                    mods = [str(m) for m in g[pre + "_mods"]]
                    out = model.forward_logits(cu(g[pre + "_y"]), {m: {} for m in mods}, cu(g[pre + "_modmask"]),
                                               return_all_logits=bool(g[pre + "_all"]))
                    assert set(out) == set(mods)
                    for m in mods:
                        ref, tol = g.expected(pre + "_logits_" + m, 2e-2)
                        assert tuple(out[m].shape) == ref.shape
                        assert float((out[m].float().cpu() - torch.from_numpy(ref)).abs().max()) < tol, (target, i, m)
    assert seen == {"forward_encoder", "forward_decoder", "forward_logits"}


def test_empty_context_decoder_needs_no_grad():
    cfg = synth.make_cfg(192, 3, 2, 2, ["tok_cam", "tok_gaze"])
    model = build_model(cfg).cuda()
    y = torch.randn(1, 10, 192, device="cuda")
    ctx = torch.zeros(1, 0, 192, device="cuda")
    with pytest.raises(NotImplementedError):
        model.forward_decoder(y, ctx, encoder_mask=torch.zeros(1, 1, 0, dtype=torch.bool, device="cuda"), decoder_attention_mask=None)
