"""CPU: the GELU / bias family (egom2p_{tiny_6e_6d,small_8e_8d,base_12e_12d}_gelu) at the drop-in boundary -- registry names,
state_dict layout derived from the reference's ego-b manifest, host-side API behaviour, the constructor's family detection,
and the oracle's family path against a plain nn.Linear / nn.LayerNorm / nn.GELU assembly. No kernel is launched here."""
import json
import os
from functools import partial

import pytest
import torch
from torch import nn

import egom2p_b200 as e
from egom2p_b200.modality_info import MODALITY_INFO as MI

import gelu_oracle as go
import synth

NAMES = ("egom2p_tiny_6e_6d_gelu", "egom2p_small_8e_8d_gelu", "egom2p_base_12e_12d_gelu")


def build(name="egom2p_base_12e_12d_gelu", mods=None, **kw):
    mods = mods or e.MOD4
    return e.create_model(name, encoder_embeddings={k: MI[k]["encoder_embedding"]() for k in mods},
                          decoder_embeddings={k: MI[k]["decoder_embedding"]() for k in mods},
                          modality_info={k: MI[k] for k in mods}, num_register_tokens=0, **kw)


@pytest.fixture(scope="module")
def base():
    torch.manual_seed(0)
    return build()


def _expected_layout(man):
    """ego-b manifest -> the GELU family's: every mlp.fc3.weight removed, fc1 / fc2 at hidden 4 * dim instead of
    2/3 * 4 * dim, a `.bias` after each biased Linear's `.weight`, LayerNorm biases become parameters under the same keys."""
    biased = ("attn.qkv.", "attn.proj.", "cross_attn.q.", "cross_attn.kv.", "cross_attn.proj.", "mlp.fc1.", "mlp.fc2.")
    sd = {}
    for k, shp in man["state_dict"].items():
        if k.endswith("mlp.fc3.weight"):
            continue
        if k.endswith("mlp.fc1.weight"):
            shp = [4 * shp[1], shp[1]]
        elif k.endswith("mlp.fc2.weight"):
            shp = [shp[0], 4 * shp[0]]
        sd[k] = shp
        if k.endswith(".weight") and any(k.endswith(b + "weight") for b in biased):
            sd[k[:-len("weight")] + "bias"] = [shp[0]]
    ln_bias = {k for k in sd if k.endswith("norm.bias") or k.endswith(("norm1.bias", "norm2.bias"))}
    params = []
    for k in man["named_parameters"]:
        if k.endswith("mlp.fc3.weight"):
            continue
        params.append(k)
        b = k[:-len("weight")] + "bias"
        if k.endswith(".weight") and (b in ln_bias or any(k.endswith(x + "weight") for x in biased)):
            params.append(b)
    return sd, params, ln_bias


def test_registry_names_resolve():
    from egom2p_b200 import registry
    for n in NAMES:
        assert registry.is_model(n)


@pytest.mark.parametrize("name,depth,dim", [("egom2p_tiny_6e_6d_gelu", 6, 384), ("egom2p_small_8e_8d_gelu", 8, 512)])
def test_small_members_dims(name, depth, dim):
    m = build(name, mods=["tok_cam", "tok_gaze"])
    assert m.gelu and len(m.encoder) == depth and len(m.decoder) == depth and m.dim == dim
    assert m.encoder[0].mlp.fc1.weight.shape == (4 * dim, dim) and not hasattr(m.encoder[0].mlp, "fc3")
    assert isinstance(m.decoder[0].context_norm.bias, nn.Parameter) and m.eps == 1e-6


def test_state_dict_follows_manifest_rule(base, golden_dir):
    man = json.load(open(os.path.join(golden_dir, "egob_state_dict_manifest.json")))
    want, params, ln_bias = _expected_layout(man)
    sd = base.state_dict()
    assert list(sd.keys()) == list(want.keys())
    assert all(list(sd[k].shape) == want[k] for k in sd)
    assert [n for n, _ in base.named_parameters()] == params
    assert len(ln_bias) == 74
    n_lin_bias = sum(1 for k in want if k.endswith(".bias") and k not in ln_bias and k != "decoder_proj_context.bias")
    assert n_lin_bias == 12 * 4 + 12 * 7
    assert sum(p.numel() for p in base.parameters()) == sum(torch.Size(want[k]).numel() for k in params)


def test_init_tying_and_no_weight_decay(base):
    for m in e.MOD4:
        dec, enc = base.decoder_embeddings[m], base.encoder_embeddings[m]
        assert dec.to_logits.weight is dec.token_emb.weight
        assert dec.mod_emb is enc.mod_emb
    assert base.no_weight_decay() == set()
    for n, p in base.named_parameters():
        if n.endswith(".bias"):
            assert float(p.detach().abs().sum()) == 0.0, n   # init_weights: Linear biases 0, LayerNorm biases 0
        elif "norm" in n and n.endswith(".weight"):
            assert bool((p == 1).all()), n
    bufs = dict(base.named_buffers())
    assert not any(k.endswith("norm1.bias") for k in bufs)   # LayerNorm biases are parameters, not buffers


def test_freeze_helpers(base):
    base.freeze_shared_params()
    assert not any(p.requires_grad for p in base.encoder.parameters())
    assert not base.decoder_norm.bias.requires_grad and not base.encoder_norm.bias.requires_grad
    assert all(p.requires_grad for p in base.encoder_embeddings.parameters())
    base.freeze_params_except_specific_embeddings("tok_rgb-tok_cam")
    assert not base.encoder_embeddings["tok_rgb"].token_emb.weight.requires_grad
    assert base.encoder_embeddings["tok_depth"].token_emb.weight.requires_grad
    base.unfreeze_all()
    assert all(p.requires_grad for p in base.parameters())


@pytest.mark.parametrize("kw", [
    dict(qkv_bias=False, proj_bias=False, mlp_bias=False, act_layer=nn.GELU, gated_mlp=False),   # GELU without biases
    dict(qkv_bias=True, proj_bias=True, mlp_bias=True, act_layer=nn.SiLU, gated_mlp=True),     # SwiGLU with biases
    dict(qkv_bias=True, act_layer=nn.GELU, gated_mlp=True),                                   # gated GELU
    dict(qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6), qk_norm=True),             # QK-norm
    dict(qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6), num_register_tokens=4),
    dict(qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6), drop_path_rate_encoder=0.1),
    dict(qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6), dim=680, num_heads=10),   # head dim 68
    dict(qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6, bias=False)),              # LayerNorm without bias
])
def test_unsupported_argument_sets_raise(kw):
    from egom2p_b200.model import EgoM2P
    mods = ["tok_cam"]
    args = dict(encoder_embeddings={k: MI[k]["encoder_embedding"]() for k in mods},
                decoder_embeddings={k: MI[k]["decoder_embedding"]() for k in mods}, modality_info={k: MI[k] for k in mods},
                dim=384, encoder_depth=1, decoder_depth=1, num_heads=6)
    args.update(kw)
    with pytest.raises(NotImplementedError):
        EgoM2P(**args)


def test_reference_arguments_build_the_family():
    from egom2p_b200.model import EgoM2P
    mods = ["tok_cam"]
    m = EgoM2P({k: MI[k]["encoder_embedding"]() for k in mods}, {k: MI[k]["decoder_embedding"]() for k in mods},
               {k: MI[k] for k in mods}, dim=384, encoder_depth=1, decoder_depth=1, num_heads=6, mlp_ratio=4, qkv_bias=True,
               norm_layer=partial(nn.LayerNorm, eps=1e-6))
    assert m.gelu and m.encoder[0].attn.qkv.bias is not None and m.decoder[0].cross_attn.proj.bias is not None


class _RefBlock(nn.Module):
    """Plain-module GELU / bias blocks (nn.Linear / nn.LayerNorm / nn.GELU), the reference's structure."""

    def __init__(self, D, H, decoder):
        super().__init__()
        ln = partial(nn.LayerNorm, eps=1e-6)
        self.H, self.decoder = H, decoder
        self.norm1, self.norm2 = ln(D), ln(D)
        self.qkv, self.proj = nn.Linear(D, 3 * D), nn.Linear(D, D)
        if decoder:
            self.query_norm, self.context_norm = ln(D), ln(D)
            self.q, self.kv, self.xproj = nn.Linear(D, D), nn.Linear(D, 2 * D), nn.Linear(D, D)
        self.fc1, self.fc2, self.act = nn.Linear(D, 4 * D), nn.Linear(4 * D, D), nn.GELU()

    def attend(self, q, k, v, mask):
        B, Nq, D = q.shape
        h, d = self.H, D // self.H
        q, k, v = (t.reshape(B, -1, h, d).transpose(1, 2) for t in (q, k, v))
        s = (q @ k.transpose(-2, -1)) * d ** -0.5
        s = s.masked_fill(mask[:, None], -torch.finfo(s.dtype).max)
        return (s.softmax(-1) @ v).transpose(1, 2).reshape(B, Nq, D)

    def forward(self, x, mask, ctx=None, xmask=None):
        D = x.shape[-1]
        qkv = self.qkv(self.norm1(x))
        x = x + self.proj(self.attend(qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:], mask))
        if self.decoder:
            kv = self.kv(self.context_norm(ctx))
            x = x + self.xproj(self.attend(self.q(self.query_norm(x)), kv[..., :D], kv[..., D:], xmask))
        return x + self.fc2(self.act(self.fc1(self.norm2(x))))


def test_oracle_family_path_matches_plain_modules():
    cfg = go.make_cfg(64, 2, 1, 1, ["tok_cam", "tok_gaze"])
    sd = go.make_state_dict(cfg, 3)
    assert float(sd["encoder.0.attn.qkv.bias"].abs().max()) > 0 and float(sd["decoder.0.norm2.bias"].abs().max()) > 0
    g = torch.Generator().manual_seed(0)
    B, N, M, D = 2, 7, 5, 64
    x, y, ctx = (torch.randn(B, n, D, generator=g) for n in (N, M, N))
    emask = torch.zeros(B, N, N, dtype=torch.bool)
    emask[1, :, 5:] = True
    dmask = torch.triu(torch.ones(M, M, dtype=torch.bool), 1)[None].expand(B, M, M)
    xmask = emask[:, :1, :].expand(B, M, N)
    enc = _RefBlock(D, 2, False)
    dec = _RefBlock(D, 2, True)
    ren = {"norm1": "norm1", "norm2": "norm2", "attn.qkv": "qkv", "attn.proj": "proj", "mlp.fc1": "fc1", "mlp.fc2": "fc2"}
    rdec = {"norm1": "norm1", "norm2": "norm2", "self_attn.qkv": "qkv", "self_attn.proj": "proj", "query_norm": "query_norm",
            "context_norm": "context_norm", "cross_attn.q": "q", "cross_attn.kv": "kv", "cross_attn.proj": "xproj",
            "mlp.fc1": "fc1", "mlp.fc2": "fc2"}
    enc.load_state_dict({f"{v}.{t}": sd[f"encoder.0.{k}.{t}"] for k, v in ren.items() for t in ("weight", "bias")})
    dec.load_state_dict({f"{v}.{t}": sd[f"decoder.0.{k}.{t}"] for k, v in rdec.items() for t in ("weight", "bias")})
    with torch.no_grad():
        torch.testing.assert_close(go.encoder_block(x, sd, "encoder.0.", emask, 2), enc(x, emask), rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(go.decoder_block(y, ctx, sd, "decoder.0.", dmask, xmask, 2), dec(y, dmask, ctx, xmask),
                                   rtol=1e-5, atol=1e-5)
        ln = nn.LayerNorm(D, eps=1e-6)
        ln.load_state_dict({"weight": sd["encoder_norm.weight"], "bias": sd["encoder_norm.bias"]})
        torch.testing.assert_close(go.forward_encoder(x, emask, sd, 1, 2), ln(enc(x, emask)), rtol=1e-5, atol=1e-5)


def test_synth_manifest_matches_model():
    cfg = go.make_cfg(384, 6, 6, 6, ["tok_cam", "tok_gaze"])
    m = build("egom2p_tiny_6e_6d_gelu", mods=["tok_cam", "tok_gaze"])
    man = go.state_dict_manifest(cfg)
    sd = m.state_dict()
    assert set(sd) == set(man) and all(tuple(sd[k].shape) == tuple(man[k]) for k in man)
    m.load_state_dict(go.make_state_dict(cfg, 1), strict=True)


@pytest.mark.skipif(not os.path.isdir("/root/reference/egom2p"), reason="the reference tree exists in the authoring container only")
def test_reference_builds_the_same_models():
    """The reference's create_model builds each GELU name with the same keys, strict load both ways, and after
    register_into_reference() the reference call returns our module."""
    from _ref_import import import_reference
    import_reference()
    from egom2p.data.modality_info import MODALITY_INFO as REF_MI
    from egom2p.utils.timm.model_builder import create_model as ref_create
    mods = ["tok_cam", "tok_gaze"]
    kw = lambda mi: dict(encoder_embeddings={m: mi[m]["encoder_embedding"]() for m in mods},
                         decoder_embeddings={m: mi[m]["decoder_embedding"]() for m in mods},
                         modality_info={m: mi[m] for m in mods}, num_register_tokens=0)
    refs = {n: ref_create(n, **kw(REF_MI)) for n in NAMES}
    for n, ref in refs.items():
        assert type(ref).__module__.startswith("egom2p.models")
        ours = e.create_model(n, **kw(MI))
        assert list(ours.state_dict().keys()) == list(ref.state_dict().keys())
        ref.load_state_dict(ours.state_dict(), strict=True)
        ours.load_state_dict(ref.state_dict(), strict=True)
    e.register_into_reference()
    model = ref_create("egom2p_tiny_6e_6d_gelu", **kw(REF_MI))
    assert type(model).__module__ == "egom2p_b200.model" and model.gelu
