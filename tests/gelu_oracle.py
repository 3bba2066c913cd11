"""TEST INFRASTRUCTURE ONLY -- the GELU / bias family (egom2p_*_gelu, egom2p_model.py:882-978) for the checks in
tests/test_gelu_family_{cpu,gpu}.py: CPU fp32 blocks and whole step (biases on every Linear and LayerNorm, MLP
fc2(GELU(fc1 x)) with nn.GELU()'s exact erf form), and synthetic configs / manifests / weights with NON-ZERO biases.

It builds on the pinned no-bias oracle (oracle/egom2p_oracle.py: index plans, attention with masked_fill(-finfo.max),
sin-cos tables) and on oracle/synth.py (batches, the weight draws of the shared keys) without changing them; only the
parts where the family differs are restated here."""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn.functional as F

import egom2p_oracle as orc
import synth


# ---------------------------------------------------------------------------------------------- synthetic configs / weights
def make_cfg(dim, heads, enc_depth, dec_depth, mods: List[str], **kw):
    """synth.make_cfg for the GELU / bias family: hidden = 4 * dim (no 2/3 gate split)."""
    cfg = synth.make_cfg(dim, heads, enc_depth, dec_depth, mods, **kw)
    cfg["hidden"] = 4 * dim
    return cfg


def state_dict_manifest(cfg) -> Dict[str, tuple]:
    """Key -> shape in the reference's state_dict layout: the no-bias family's (synth.state_dict_manifest) with every
    mlp.fc3.weight removed and a `.bias` after each Linear's `.weight` (LayerNorm biases keep their keys)."""
    biased = ("attn.qkv.", "attn.proj.", "cross_attn.q.", "cross_attn.kv.", "cross_attn.proj.", "mlp.fc1.", "mlp.fc2.")
    man: Dict[str, tuple] = {}
    for k, shp in synth.state_dict_manifest(cfg).items():
        if k.endswith("mlp.fc3.weight"):
            continue
        man[k] = shp
        if any(k.endswith(b + "weight") for b in biased):
            man[k[:-len("weight")] + "bias"] = (shp[0],)
    return man


def make_state_dict(cfg, seed: int, tie: bool = True) -> Dict[str, torch.Tensor]:
    """Random weights with the draws of synth.make_state_dict for the shared kinds of tensor, and every bias non-zero:
    Linears N(0, 0.02), LayerNorms N(0, 0.1) -- the reference init (all zero) would hide every bias bug."""
    rng = np.random.default_rng(seed)
    sd: Dict[str, torch.Tensor] = {}
    for k, shp in state_dict_manifest(cfg).items():
        if k.endswith("pos_emb"):
            inf = cfg["mods"][k.split(".")[1]]
            tab = orc.sincos_3d(*inf["thw"], cfg["dim"]) if "thw" in inf else orc.sincos_1d(inf["len"], cfg["dim"])
            sd[k] = tab[None].clone()
        elif k.endswith("to_logits.weight"):
            continue
        elif k.endswith(".bias"):
            sd[k] = torch.from_numpy(((0.1 if "norm" in k else 0.02) * rng.standard_normal(shp)).astype(np.float32))
        elif "norm" in k and k.endswith(".weight"):
            sd[k] = torch.from_numpy((1.0 + 0.1 * rng.standard_normal(shp)).astype(np.float32))
        elif len(shp) == 2 and "token_emb" not in k:
            b = math.sqrt(6.0 / (shp[0] + shp[1]))
            sd[k] = torch.from_numpy(rng.uniform(-b, b, shp).astype(np.float32))
        else:
            sd[k] = torch.from_numpy((0.02 * rng.standard_normal(shp)).astype(np.float32))
    for m in cfg["mods"]:
        p = f"decoder_embeddings.{m}."
        sd[p + "mod_emb"] = sd[f"encoder_embeddings.{m}.mod_emb"]
        if tie:
            sd[p + "to_logits.weight"] = sd[p + "token_emb.weight"]
        else:
            shp = sd[p + "token_emb.weight"].shape
            b = math.sqrt(6.0 / (shp[0] + shp[1]))
            sd[p + "to_logits.weight"] = torch.from_numpy(rng.uniform(-b, b, tuple(shp)).astype(np.float32))
    return sd


# ---------------------------------------------------------------------------------------------- blocks
def _ln(x, sd, pre, eps=1e-6):
    return F.layer_norm(x, (x.shape[-1],), sd[pre + "weight"], sd[pre + "bias"], eps)


def _lin(x, sd, pre):
    return F.linear(x, sd[pre + "weight"], sd[pre + "bias"])


def _mlp(x, sd, pre):
    return _lin(F.gelu(_lin(x, sd, pre + "fc1.")), sd, pre + "fc2.")


def encoder_block(x, sd, pre, mask, heads):
    D = x.shape[-1]
    qkv = _lin(_ln(x, sd, pre + "norm1."), sd, pre + "attn.qkv.")
    x = x + _lin(orc._attend(qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:], mask, heads), sd, pre + "attn.proj.")
    return x + _mlp(_ln(x, sd, pre + "norm2."), sd, pre + "mlp.")


def decoder_block(y, ctx, sd, pre, sa_mask, xa_mask, heads):
    """An empty context (N = 0) gives a zero cross-attention output, so that sub-block adds the projection's bias."""
    D = y.shape[-1]
    qkv = _lin(_ln(y, sd, pre + "norm1."), sd, pre + "self_attn.qkv.")
    y = y + _lin(orc._attend(qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:], sa_mask, heads), sd, pre + "self_attn.proj.")
    q = _lin(_ln(y, sd, pre + "query_norm."), sd, pre + "cross_attn.q.")
    kv = _lin(_ln(ctx, sd, pre + "context_norm."), sd, pre + "cross_attn.kv.")
    y = y + _lin(orc._attend(q, kv[..., :D], kv[..., D:], xa_mask, heads), sd, pre + "cross_attn.proj.")
    return y + _mlp(_ln(y, sd, pre + "norm2."), sd, pre + "mlp.")


def forward_encoder(x, enc_mask, sd, depth, heads):
    for i in range(depth):
        x = encoder_block(x, sd, f"encoder.{i}.", enc_mask, heads)
    return _ln(x, sd, "encoder_norm.")


def forward_decoder(y, ctx, enc_mask, dec_attn_mask, sd, depth, heads):
    for i in range(depth):
        y = decoder_block(y, ctx, sd, f"decoder.{i}.", dec_attn_mask, enc_mask, heads)
    return _ln(y, sd, "decoder_norm.")


# ---------------------------------------------------------------------------------------------- whole step
def forward(sd: Dict[str, torch.Tensor], cfg: dict, mod_dict, num_encoder_tokens: int, num_decoder_tokens: int,
            dec_order: Optional[List[str]] = None, return_logits: bool = False, keep: bool = False):
    """egom2p_oracle.forward with the family's blocks ('mod' loss): same index plans, gathers and heads."""
    heads, D = cfg["heads"], cfg["dim"]
    mods = [m for m in mod_dict if m in cfg["mods"]]
    mod_ids = {m: cfg["mods"][m]["id"] for m in mods}
    B = mod_dict[mods[0]]["tensor"].shape[0]
    dec_order = dec_order or mods
    ep = orc.plan_encoder({m: mod_dict[m]["input_mask"].numpy() for m in mods}, mod_ids, num_encoder_tokens)
    xs, es = [], []
    for m in mods:
        ids = mod_dict[m]["tensor"].reshape(B, -1).long()
        pre = f"encoder_embeddings.{m}."
        xs.append(sd[pre + "token_emb.weight"][ids])
        es.append((sd[pre + "pos_emb"] + sd[pre + "mod_emb"]).expand(B, -1, -1))
    keep_e = torch.from_numpy(ep["ids_keep"])[..., None].expand(-1, -1, D)
    emask = torch.from_numpy(ep["mask"])
    enc_tok = torch.gather(torch.cat(xs, 1), 1, keep_e).masked_fill(emask[..., None], 0.0)
    enc_emb = torch.gather(torch.cat(es, 1), 1, keep_e).masked_fill(emask[..., None], 0.0)
    dp = orc.plan_decoder({m: mod_dict[m]["target_mask"].numpy() for m in mods},
                          {m: mod_dict[m]["decoder_attention_mask"].numpy() for m in mods},
                          {m: mod_dict[m]["tensor"].reshape(B, -1).numpy() for m in mods},
                          mod_ids, dec_order, num_decoder_tokens, causal=cfg.get("causal", False), sep=cfg.get("sep", True))
    es = [(sd[f"decoder_embeddings.{m}.pos_emb"] + sd[f"decoder_embeddings.{m}.mod_emb"]).expand(B, -1, -1) for m in dec_order]
    keep_d = torch.from_numpy(dp["ids_keep"])[..., None].expand(-1, -1, D)
    dmask = torch.from_numpy(dp["mask"])
    dec_emb = torch.gather(torch.cat(es, 1), 1, keep_d)
    y0 = ((torch.zeros_like(dec_emb) + sd["mask_token"]) + dec_emb).masked_fill(dmask[..., None], 0.0)
    enc_mask3 = emask[:, None, :]
    x = forward_encoder(enc_tok + enc_emb, enc_mask3, sd, cfg["enc_depth"], heads)
    ctx = F.linear(x, sd["decoder_proj_context.weight"], sd["decoder_proj_context.bias"]) + enc_emb
    y = forward_decoder(y0, ctx, enc_mask3, torch.from_numpy(dp["attn_mask"]), sd, cfg["dec_depth"], heads)
    out = {"dec_plan": dp} if keep else {}
    if return_logits:
        out["logits"] = {m: F.linear(y, sd[f"decoder_embeddings.{m}.to_logits.weight"]) for m in mods}
        return out
    dec_mod = torch.from_numpy(dp["mod_mask"].astype(np.int64))
    tgt = torch.from_numpy(dp["target_ids"])
    mod_loss = {}
    for m in mods:
        sel = dec_mod == mod_ids[m]
        logits = F.linear(y[sel], sd[f"decoder_embeddings.{m}.to_logits.weight"])
        mod_loss[m] = logits.sum() if logits.numel() == 0 else F.cross_entropy(logits, tgt[sel], reduction="mean")
    out["loss"], out["mod_loss"] = sum(mod_loss.values()) / len(mod_loss), mod_loss
    return out
