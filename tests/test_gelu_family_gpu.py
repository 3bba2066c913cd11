"""GPU: the GELU / bias family (egom2p_*_gelu) on the sm_100a kernels. Kernel level against torch fp32 on the same bf16
operands (LayerNorm with bias, bf16-output GEMM with bias, GELU forward / backward epilogues, bias-gradient column sums);
model level against the CPU oracle with non-zero biases everywhere (dense, packed ragged and slot-layout ragged batches,
tolerances as tests/test_model_gpu.py, bias and LayerNorm-bias gradients included); a 3-step AdamW trajectory; one CUDA-graph
capture; the generation sampler's guided step and a full guided rgb -> cam generation; one base-dims dense case."""
import random
from functools import partial

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

pytestmark = pytest.mark.gpu

import gelu_oracle as go  # noqa: E402
import synth  # noqa: E402

bf16, f32 = torch.bfloat16, torch.float32
MODS4 = ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"]


def _rel(a, b):
    return float((a.float().cpu() - b.float().cpu()).norm() / (b.float().cpu().norm() + 1e-12))


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("R,dim", [pytest.param(1000, 384, id="384"), pytest.param(1000, 768, id="768"), (34751, 768), (1, 768)])
def test_layernorm_bias_fwd_bwd(R, dim):
    from egom2p_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(R, dim, device="cuda", generator=g) * 2 + 0.5
    w = 1 + 0.1 * torch.randn(dim, device="cuda", generator=g)
    b = 0.1 * torch.randn(dim, device="cuda", generator=g)
    dy = torch.randn(R, dim, device="cuda", generator=g)
    dx_in = torch.randn(R, dim, device="cuda", generator=g)
    yb, yf, mean, rstd = ops.layernorm_fwd(x, w, 1e-6, out_bf16=True, out_f32=True, bias=b)
    xr, wr, br = (t.detach().clone().requires_grad_(True) for t in (x, w, b))
    ref = F.layer_norm(xr, (dim,), wr, br, 1e-6)
    assert float((yf - ref.detach()).abs().max()) < 1e-4
    assert float((yb.float() - ref.detach()).abs().max()) < 2e-2
    ref.backward(dy)
    dw, db = torch.zeros(dim, device="cuda"), torch.zeros(dim, device="cuda")
    for dyv in (dy, dy.to(bf16)):
        dw.zero_(); db.zero_()
        dx, _ = ops.layernorm_bwd(dyv, x, w, mean, rstd, dx_in=dx_in, d_weight=dw, d_bias=db)
        tol = 1e-4 if dyv.dtype == f32 else 1e-2
        assert _rel(dx, xr.grad + dx_in) < tol and _rel(dw, wr.grad) < tol and _rel(db, br.grad) < tol


@pytest.mark.parametrize("M,N,K", [(300, 2304, 768), (4096, 1152, 384), (77, 768, 512)])
def test_gemm_bf16_output_with_bias(M, N, K):
    from egom2p_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(M, K, device="cuda", generator=g).to(bf16)
    w = (torch.randn(N, K, device="cuda", generator=g) * K ** -0.5).to(bf16)
    b = torch.randn(N, device="cuda", generator=g)
    y = ops.linear_fwd(x, w, bias=b)
    ref = x.float() @ w.float().t() + b
    assert y.dtype == bf16 and float((y.float() - ref).abs().max()) < 2e-2 * float(ref.abs().max())
    assert float((ops.linear_fwd(x, w).float() - (ref - b)).abs().max()) < 2e-2 * float(ref.abs().max())   # no-bias path unchanged


def test_gelu_epilogues_sweep():
    """u = x W1^T + b1 swept over |u| up to ~8; GELU(u) and du = dh * GELU'(u) against torch fp32 (exact erf GELU)."""
    from egom2p_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(2)
    M, K, N, D = 1000, 384, 1536, 384
    x = torch.randn(M, K, device="cuda", generator=g).to(bf16)
    w1 = (torch.randn(N, K, device="cuda", generator=g) * 3 * K ** -0.5).to(bf16)   # |acc| ~ 3 sigma: tails past 8
    b1 = torch.linspace(-4, 4, N, device="cuda")
    u, h = ops.gemm_gelu_fwd(x, w1, b1)
    uref = x.float() @ w1.float().t() + b1
    assert float(uref.abs().max()) > 8
    assert float((u.float() - uref).abs().max()) < 1e-2 * float(uref.abs().max())
    href = F.gelu(uref)
    assert float(((h.float() - href).abs() / (href.abs() + 1e-2)).max()) < 2e-2
    dy = torch.randn(M, D, device="cuda", generator=g).to(bf16)
    w2 = (torch.randn(D, N, device="cuda", generator=g) * N ** -0.5).to(bf16)
    du = ops.gemm_gelu_bwd(dy, w2, u)
    uu = u.float().requires_grad_(True)
    F.gelu(uu).backward(dy.float() @ w2.float())
    assert _rel(du, uu.grad) < 1e-2
    assert float((du.float() - uu.grad).abs().max()) < 2e-2 * float(uu.grad.abs().max())


@pytest.mark.parametrize("rows,cols", [(65536, 2304), (65536, 768), (333, 1536), (34751, 2304), (1, 768)])
def test_bias_grad_colsum(rows, cols):
    from egom2p_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    full = torch.randn(rows, cols + 64, device="cuda", generator=g).to(bf16)
    x = full[:, 16:16 + cols]                                  # a strided view, as the qkv / kv slices are
    out = torch.full((cols,), 1.0, device="cuda")
    ops.colsum_bf16(x, out)
    ref = x.double().sum(0) + 1.0
    assert float((out.double() - ref).abs().max()) < 1e-4 * rows ** 0.5 * 4


# ------------------------------------------------------------------------------------------------ model
def build_gelu(cfg, tie=True):
    from egom2p_b200 import adapters as A
    from egom2p_b200.model import EgoM2P
    enc, dec, info = {}, {}, {}
    for m, inf in cfg["mods"].items():
        if "thw" in inf:
            isz = inf["thw"][1] * 8
            enc[m] = A.VideoTokenEncoderEmbedding(vocab_size=inf["vocab"], image_size=isz)
            dec[m] = A.VideoTokenDecoderEmbedding(vocab_size=inf["vocab"], image_size=isz, share_embedding=tie)
        else:
            enc[m] = A.GazeCamTokenEncoderEmbedding(vocab_size=inf["vocab"])
            dec[m] = A.GazeCamTokenDecoderEmbedding(vocab_size=inf["vocab"], share_embedding=tie)
        info[m] = {"id": inf["id"], "vocab_size": inf["vocab"], "type": inf["type"], "max_tokens": inf["len"]}
    return EgoM2P(enc, dec, info, dim=cfg["dim"], encoder_depth=cfg["enc_depth"], decoder_depth=cfg["dec_depth"],
                  num_heads=cfg["heads"], mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6))


def to_cuda(md):
    return {m: {k: v.cuda() for k, v in d.items()} for m, d in md.items()}


def _leaves(sd, cfg):
    leaf = {}
    for k, v in sd.items():
        if k.endswith("to_logits.weight") or (k.startswith("decoder_embeddings") and k.endswith("mod_emb")):
            continue
        leaf[k] = v.clone().requires_grad_(v.is_floating_point() and not k.endswith("pos_emb"))
    for m in cfg["mods"]:
        leaf[f"decoder_embeddings.{m}.to_logits.weight"] = leaf[f"decoder_embeddings.{m}.token_emb.weight"]
        leaf[f"decoder_embeddings.{m}.mod_emb"] = leaf[f"encoder_embeddings.{m}.mod_emb"]
    return leaf


def check_case(cfg, md, n_enc, n_dec, seed, shuffle_seed, pack_rows=True, logits=True):
    sd = go.make_state_dict(cfg, seed)
    model = build_gelu(cfg).cuda()
    model.load_state_dict(sd, strict=True)
    model.pack_rows = pack_rows
    mods = list(cfg["mods"])
    random.seed(shuffle_seed)
    order = random.sample(mods, len(mods))
    leaf = _leaves(sd, cfg)
    ref = go.forward(leaf, cfg, md, n_enc, n_dec, dec_order=order, keep=True)
    ref["loss"].backward()
    random.seed(shuffle_seed)
    loss, mod_loss = model(to_cuda(md), n_enc, n_dec)
    loss.backward()
    torch.cuda.synchronize()
    rel = abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item())
    assert rel < 1e-3, f"loss {loss.item()} vs oracle {ref['loss'].item()} (rel {rel})"
    bad, n_bias = [], 0
    for name, p in model.named_parameters():
        g_ref = leaf[name].grad
        if g_ref is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name
            continue
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
        n_bias += name.endswith(".bias")
        err = _rel(p.grad, g_ref)
        tol = 5e-2 if ("cross_attn.q." in name or "query_norm" in name) else 3e-2
        if err > tol:
            bad.append((name, err))
    assert not bad, bad
    assert n_bias > 0
    if logits:
        with torch.no_grad():
            random.seed(shuffle_seed)
            lg = model(to_cuda(md), n_enc, n_dec, return_logits=True)
            lo = go.forward(sd, cfg, md, n_enc, n_dec, dec_order=order, return_logits=True)["logits"]
        valid = torch.from_numpy(~ref["dec_plan"]["mask"])
        for m in mods:
            diff = (lg[m].float().cpu() - lo[m])[valid].abs().max().item() if valid.any() else 0.0
            assert diff < 2e-2, f"logits {m}: max-abs {diff}"
    return model


def _tiny_cfg():
    return go.make_cfg(384, 6, 2, 2, MODS4, video_vocab=512, video_thw=(5, 4, 4))


RAGGED = dict(n_in={"tok_cam": [5, 1, 30, 2], "tok_depth": [30, 10, 0, 1], "tok_gaze": [4, 0, 30, 0], "tok_rgb": [25, 40, 4, 3]},
              n_tgt={"tok_cam": [10, 30, 0, 1], "tok_depth": [20, 0, 40, 0], "tok_gaze": [3, 0, 0, 0], "tok_rgb": [15, 18, 70, 4]})


def test_step_dense():
    cfg = go.make_cfg(384, 6, 2, 2, MODS4, video_vocab=1024, video_thw=(5, 8, 8))
    B = 2
    md = synth.make_batch(cfg, B=B, seed=3, n_in={"tok_cam": [15] * B, "tok_depth": [145] * B, "tok_gaze": [15] * B, "tok_rgb": [145] * B},
                          n_tgt={"tok_cam": [15] * B, "tok_depth": [145] * B, "tok_gaze": [15] * B, "tok_rgb": [145] * B})
    check_case(cfg, md, 320, 320, seed=9, shuffle_seed=1)


@pytest.mark.parametrize("pack_rows", [True, False])
def test_step_ragged(pack_rows):
    cfg = _tiny_cfg()
    md = synth.make_batch(cfg, B=4, seed=11, **RAGGED)
    check_case(cfg, md, 64, 48, seed=5, shuffle_seed=3, pack_rows=pack_rows)


def test_adamw_trajectory_follows_oracle():
    from egom2p_b200.optim import FusedAdamW
    cfg = _tiny_cfg()
    md = synth.make_batch(cfg, B=4, seed=12, **RAGGED)
    sd = go.make_state_dict(cfg, 6)
    mods = list(cfg["mods"])
    orders = []
    for s in range(3):
        random.seed(100 + s)
        orders.append(random.sample(mods, len(mods)))
    lr = 3e-3
    leaf = _leaves(sd, cfg)
    params = list({id(t): t for t in leaf.values() if t.requires_grad}.values())
    opt = torch.optim.AdamW(params, lr=lr, betas=(0.9, 0.95), weight_decay=0.05)
    ref = []
    for order in orders:
        out = go.forward(leaf, cfg, md, 64, 48, dec_order=order)
        out["loss"].backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
        ref.append(out["loss"].item())
    model = build_gelu(cfg).cuda()
    model.load_state_dict(sd, strict=True)
    params = [p for p in model.parameters() if p.requires_grad]
    opt = FusedAdamW([{"params": params, "weight_decay": 0.05}], lr=lr, betas=(0.9, 0.95))
    mdc = to_cuda(md)
    got = []
    for s in range(3):
        random.seed(100 + s)
        loss, _ = model(mdc, 64, 48)
        loss.backward()
        opt.clip_grad_norm_(1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
        got.append(loss.item())
    assert ref[0] - ref[-1] > 0.02 * ref[0], ref
    for s, (a, b) in enumerate(zip(got, ref)):
        tol = 1e-3 if s == 0 else 1.5e-2
        assert abs(a - b) / abs(b) < tol, f"step {s}: {got} vs oracle {ref}"


def test_graphed_step_matches_eager():
    from egom2p_b200.graphed import GraphedTrainStep
    from egom2p_b200.optim import FusedAdamW
    cfg = _tiny_cfg()
    n_in = {"tok_cam": [5, 30], "tok_depth": [30, 10], "tok_gaze": [4, 3], "tok_rgb": [25, 21]}
    n_tg = {"tok_cam": [10, 3], "tok_depth": [20, 7], "tok_gaze": [3, 7], "tok_rgb": [15, 18]}
    batches = [to_cuda(synth.make_batch(cfg, B=2, seed=30 + i, n_in=n_in, n_tgt=n_tg)) for i in range(2)]
    sd = go.make_state_dict(cfg, 7)
    models = []
    for _ in range(2):
        m = build_gelu(cfg).cuda()
        m.load_state_dict(sd, strict=True)
        models.append(m)
    eager, graphed = models
    mk = lambda m: FusedAdamW([{"params": [p for p in m.parameters() if p.requires_grad], "weight_decay": 0.05}], lr=1e-3,
                              betas=(0.9, 0.95))
    o_e, o_g = mk(eager), mk(graphed)
    runner = GraphedTrainStep(graphed, o_g, batches[1], 64, 48, clip_grad=1.0)
    eager.fixed_decoder_order = list(graphed.fixed_decoder_order)
    loss_e, _ = eager(batches[0], 64, 48)
    loss_e.backward()
    o_e.clip_grad_norm_(1.0)
    o_e.step()
    loss_g = runner(batches[0])
    torch.cuda.synchronize()
    assert abs(loss_e.item() - loss_g.item()) <= 2e-4 * abs(loss_e.item()), (loss_e.item(), loss_g.item())


def test_base_dims_dense_against_oracle():
    """egom2p_base_12e_12d_gelu block dims (dim 768, 12 heads, hidden 3072) on a 1 + 1 layer model, b = 1, N = M = 2048."""
    cfg = go.make_cfg(768, 12, 1, 1, ["tok_depth", "tok_rgb"], video_vocab=1024, video_thw=(5, 24, 24))
    md = synth.make_batch(cfg, B=1, seed=4, n_in={"tok_depth": [1024], "tok_rgb": [1024]}, n_tgt={"tok_depth": [1024], "tok_rgb": [1024]})
    check_case(cfg, md, 2048, 2048, seed=2, shuffle_seed=0, logits=False)


# ------------------------------------------------------------------------------------------------ sampler
def _sampler():
    from egom2p_b200.generate import GenerationSampler
    cfg = _tiny_cfg()
    model = build_gelu(cfg).cuda().eval()
    sd = go.make_state_dict(cfg, 3)
    model.load_state_dict(sd, strict=True)
    return GenerationSampler(model), cfg, sd


def test_forward_hidden_guided_step_against_oracle():
    s, cfg, sd = _sampler()
    rng = np.random.default_rng(0)
    B, L, k = 1, 80, 5
    ids = rng.integers(0, 512, (B, L))
    md = {"tok_rgb": {"tensor": torch.from_numpy(ids.reshape(B, 5, 4, 4)).cuda(), "input_mask": torch.zeros(B, L, dtype=torch.bool).cuda(),
                      "target_mask": torch.ones(B, L, dtype=torch.bool).cuda()},
          "tok_cam": {"tensor": torch.zeros(B, 30, dtype=torch.int64).cuda(), "input_mask": torch.ones(B, 30, dtype=torch.bool).cuda(),
                      "target_mask": torch.zeros(B, 30, dtype=torch.bool).cuda()}}
    pos = torch.tensor([[7, 11, 29, 5, 20]]).cuda()
    with torch.no_grad():
        yn = s.forward_hidden(md, "tok_cam", ["tok_rgb"], {"tok_rgb": [L], "tok_cam": [0]}, pos).reshape(2, B, k, -1)
    # oracle: encoder over every rgb token, context projection, decoder over the k masked cam positions; the unconditional
    # branch has no context at all (its cross-attention output is 0 and only the projection's bias remains)
    D = cfg["dim"]
    e = "encoder_embeddings.tok_rgb."
    x = sd[e + "token_emb.weight"][torch.from_numpy(ids)] + sd[e + "pos_emb"] + sd[e + "mod_emb"]
    enc = go.forward_encoder(x, None, sd, cfg["enc_depth"], cfg["heads"])
    ctx = F.linear(enc, sd["decoder_proj_context.weight"], sd["decoder_proj_context.bias"]) + sd[e + "pos_emb"] + sd[e + "mod_emb"]
    d = "decoder_embeddings.tok_cam."
    y0 = sd["mask_token"] + sd[d + "pos_emb"][:, pos[0].cpu()] + sd[d + "mod_emb"]
    head = sd[d + "to_logits.weight"]
    for branch, c in ((0, ctx), (1, torch.zeros(B, 0, D))):
        ref = go.forward_decoder(y0, c, None, None, sd, cfg["dec_depth"], cfg["heads"])
        diff = float((F.linear(yn[branch].cpu(), head) - F.linear(ref, head)).abs().max())
        assert diff < 2e-2, (branch, diff)


def test_decoder_without_context_against_oracle():
    """No context token in any sample (the sampler's call when no branch has conditioning): forward_decoder with N = 0 and
    decode_tokens(y0, None, None). Each cross-attention then adds only its projection's bias."""
    s, cfg, sd = _sampler()
    B, k, D = 2, 5, cfg["dim"]
    d = "decoder_embeddings.tok_cam."
    pos = torch.tensor([[7, 11, 29, 5, 20], [0, 3, 4, 17, 28]])
    y0 = sd["mask_token"] + sd[d + "pos_emb"][0, pos] + sd[d + "mod_emb"]
    ref = go.forward_decoder(y0, torch.zeros(B, 0, D), None, None, sd, cfg["dec_depth"], cfg["heads"])
    with torch.no_grad():
        got = {"forward_decoder": s.model.forward_decoder(y0.cuda(), torch.zeros(B, 0, D, device="cuda"), None, None),
               "decode_tokens": s.model.decode_tokens(y0.cuda(), None, None).reshape(B, k, D)}
    head = sd[d + "to_logits.weight"]
    for name, yn in got.items():
        diff = float((F.linear(yn.cpu(), head) - F.linear(ref, head)).abs().max())
        assert diff < 2e-2, (name, diff)


def test_generate_rgb_to_cam_guided():
    from egom2p_b200.generate import build_chained_generation_schedules, init_empty_target_modality, init_full_input_modality
    s, cfg, _ = _sampler()
    info = s.model.modality_info
    B = 2
    rng = np.random.default_rng(1)
    md = {"tok_rgb": {"tensor": torch.from_numpy(rng.integers(0, 512, (B, 5, 4, 4))).cuda()}}
    md = init_empty_target_modality(md, info, "tok_cam", B, 30, "cuda")
    md = init_full_input_modality(md, info, "tok_rgb", "cuda")
    schedule = build_chained_generation_schedules(
        cond_domains=["tok_rgb"], target_domains=["tok_cam"], tokens_per_target=[30], autoregression_schemes=["roar"],
        decoding_steps=[3], token_decoding_schedules=["linear"], temps=[1.0], temp_schedules=["constant"], cfg_scales=[2.0],
        cfg_schedules=["constant"], cfg_grow_conditioning=True)
    out = s.generate(md, schedule, top_p=0.8, top_k=0.0, seed=0)
    assert bool(out["tok_cam"]["target_mask"].all()) and not bool(out["tok_cam"]["input_mask"].any())
    assert 0 <= int(out["tok_cam"]["tensor"].min()) and int(out["tok_cam"]["tensor"].max()) < 256
