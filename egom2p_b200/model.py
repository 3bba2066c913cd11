"""Drop-in replacement of the reference `EgoM2P` module (egom2p/models/egom2p_model.py:57-819) whose forward /
backward run on the sm_100a kernels of libegom2p_b200.so.

Boundary kept intact: constructor signature, `forward(mod_dict, num_encoder_tokens, num_decoder_tokens, loss_type,
return_logits)`, the masking-dict layout, adapter objects (reference adapters work, duck-typed), parameter / buffer
names and shapes (strict `load_state_dict` of reference checkpoints), `forward_encoder / forward_decoder /
forward_logits / decoder_proj_context / mask_token / cat_encoder_tensors` for the GenerationSampler, freeze helpers,
`no_weight_decay`. What changed is *how* the step is computed (SURVEY.md section 7): index plan + fused embed/gather,
range-masked flash attention, tcgen05 GEMMs with fused epilogues, vocabulary head fused with cross-entropy.
Autograd nodes are per block, so DDP's bucketed all-reduce overlaps with backward exactly as for the reference.

Scope: the swiglu / no-bias family (ego-b and its tiny/small siblings) and the GELU / bias family (egom2p_*_gelu: biases
on every Linear and LayerNorm, MLP fc2(GELU(fc1 x)), egom2p_model.py:882-978), both at head dim 64. Other registered
variants of the reference (QK-norm, large / xlarge) are not built here and raise NotImplementedError at construction.
"""
from __future__ import annotations

import math
import random
from functools import partial
from typing import Any, Dict, List, Optional, Union

import torch
from torch import nn

from . import ops

bf16, f32 = torch.bfloat16, torch.float32


# =============================================================================================== parameter containers
class LayerNorm(nn.Module):
    """Parameter container mirroring egom2p_utils.LayerNorm (weight + zero `bias` buffer when bias=False) and, with
    bias=True, nn.LayerNorm (weight + `bias` Parameter) of the GELU / bias family."""

    def __init__(self, normalized_shape: int, eps=1e-5, bias=True):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(normalized_shape))
        if bias:
            self.bias = nn.Parameter(torch.zeros(normalized_shape))
        else:
            self.register_buffer("bias", torch.zeros(normalized_shape))
        self.normalized_shape = (normalized_shape,)

    def forward(self, x):
        shape = x.shape
        _, y, _, _ = ops.layernorm_fwd(x.reshape(-1, shape[-1]).float().contiguous(), self.weight.detach(), self.eps,
                                       out_bf16=False, out_f32=True, save_stats=False, bias=_det(_bias(self)))
        return y.reshape(shape)


def _bias(m: nn.Module) -> Optional[torch.Tensor]:
    """The learnable bias of a Linear or LayerNorm, None when it has none (the no-bias family's LayerNorms hold a zero buffer)."""
    return m.bias if isinstance(m.bias, nn.Parameter) else None


def _weights_and_biases(*mods: nn.Module) -> List[Optional[torch.Tensor]]:
    """weight, bias (or None) of each module in turn: the flat parameter list the block functions take."""
    return [t for m in mods for t in (m.weight, _bias(m))]


def _det(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    return None if t is None else t.detach()


class _Linear(nn.Linear):
    """nn.Linear container. Standalone calls (the sampler uses `decoder_proj_context(x)`) run the tcgen05 GEMM."""

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        shape = x.shape
        x2 = x.reshape(-1, shape[-1])
        xb = x2 if x2.dtype == bf16 else ops.cast_bf16(x2.float().contiguous())
        y = ops.linear_fwd(xb, ops.cached_bf16(self.weight), bias=None if self.bias is None else self.bias.detach(), out_dtype=f32)
        return y.reshape(*shape[:-1], -1)


# The MLP is the only part of a block that differs between the two families. Each MLP container owns, for the shared block
# code: params() -- its parameters, in the order the block functions take them; operands() -- their cached bf16 GEMM
# operands; fwd() -- x1 + MLP(h2) from the normed h2, and what bwd() needs; bwd() -- dh2 and the gradients of params(), None
# for each parameter whose flag in `need` is False (a frozen parameter gets neither its wgrad GEMM nor its bias column sum).
class GatedMlp(nn.Module):
    """fc2(SiLU(fc1 x) * fc3 x) without biases (the swiglu / no-bias family). fc1 and fc3 run as one GEMM over an operand
    with their rows interleaved (EgoM2P._bf16), the gate in its epilogue."""

    def __init__(self, dim, hidden):
        super().__init__()
        hidden = int(2 * hidden / 3)
        self.fc1 = _Linear(dim, hidden, bias=False)
        self.fc2 = _Linear(hidden, dim, bias=False)
        self.fc3 = _Linear(dim, hidden, bias=False)

    def params(self):
        return self.fc1.weight, self.fc2.weight, self.fc3.weight

    def operands(self, cache, key):
        return cache((*key, "w13"), self.fc1.weight, self.fc3.weight), cache((*key, "w2"), self.fc2.weight, pad32=True)

    def fwd(self, h2, x1, w, params):
        w13, w2 = w
        ab, g = ops.gemm_swiglu_fwd(h2, w13)   # fc1|fc3 GEMM with the SwiGLU gate in its epilogue
        return ops.linear_fwd(g, w2, addend=x1, out_dtype=f32), (ab, g)

    def bwd(self, dx2b, h2, w, saved, need):
        (w13, w2), (ab, g) = w, saved
        n1, n2, n3 = need
        dw2 = ops.linear_wgrad(dx2b, g) if n2 else None
        dab = ops.gemm_swiglu_bwd(dx2b, w2, ab)   # fc2 dgrad with the SwiGLU derivative in its epilogue
        dw13 = ops.linear_wgrad(dab, h2) if (n1 or n3) else None   # one interleaved GEMM for fc1 and fc3
        dh2 = ops.linear_dgrad(dab, w13)
        F = self.fc1.out_features
        d1, d3 = _split_w13_grad(dw13, F) if dw13 is not None else (None, None)
        return dh2, (d1 if n1 else None, dw2[:, :F] if n2 else None, d3 if n3 else None)


class Mlp(nn.Module):
    """fc2(GELU(fc1 x)) with biases (egom2p_utils.py Mlp, the GELU / bias family)."""

    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = _Linear(dim, hidden, bias=True)
        self.fc2 = _Linear(hidden, dim, bias=True)

    def params(self):
        return self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias

    def operands(self, cache, key):
        return cache((*key, "w1"), self.fc1.weight), cache((*key, "w2"), self.fc2.weight, pad32=True)

    def fwd(self, h2, x1, w, params):
        (w1, w2), (_, b1, _, b2) = w, params
        u, a = ops.gemm_gelu_fwd(h2, w1, b1)   # fc1 GEMM with + b1 and GELU in its epilogue
        return ops.linear_fwd(a, w2, bias=b2, addend=x1, out_dtype=f32), (u, a)

    def bwd(self, dx2b, h2, w, saved, need):
        (w1, w2), (u, a) = w, saved
        n1, nb1, n2, nb2 = need
        dw2 = ops.linear_wgrad(dx2b, a) if n2 else None
        db2 = ops.colsum_bf16(dx2b) if nb2 else None
        du = ops.gemm_gelu_bwd(dx2b, w2, u)   # fc2 dgrad with GELU'(u) in its epilogue
        dw1 = ops.linear_wgrad(du, h2) if n1 else None
        db1 = ops.colsum_bf16(du) if nb1 else None
        return ops.linear_dgrad(du, w1), (dw1, db1, dw2, db2)


class Attention(nn.Module):
    def __init__(self, dim, num_heads, bias=False):
        super().__init__()
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = _Linear(dim, dim * 3, bias=bias)
        self.proj = _Linear(dim, dim, bias=bias)


class CrossAttention(nn.Module):
    def __init__(self, dim, num_heads, bias=False):
        super().__init__()
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.q = _Linear(dim, dim, bias=bias)
        self.kv = _Linear(dim, dim * 2, bias=bias)
        self.proj = _Linear(dim, dim, bias=bias)


class Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio, norm_layer, gelu=False):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.attn = Attention(dim, num_heads, bias=gelu)
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp(dim, int(dim * mlp_ratio)) if gelu else GatedMlp(dim, int(dim * mlp_ratio))


class DecoderBlock(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio, norm_layer, gelu=False):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.self_attn = Attention(dim, num_heads, bias=gelu)
        self.cross_attn = CrossAttention(dim, num_heads, bias=gelu)
        self.query_norm = norm_layer(dim)
        self.context_norm = norm_layer(dim)
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp(dim, int(dim * mlp_ratio)) if gelu else GatedMlp(dim, int(dim * mlp_ratio))


# =============================================================================================== kernels glue
class _Geom:
    """Shapes + key-range tables of one forward (device tensors, no host syncs)."""
    __slots__ = ("B", "N", "M", "H", "D", "enc_lo", "enc_hi", "dec_lo", "dec_hi", "x_lo", "x_hi", "eps", "m_enc", "m_dec", "m_x",
                 "ctx_users", "dctx_acc", "epoch_ref", "p_enc", "p_dec", "p_x")

    def build_meta(self, dev, encoder: bool = True):
        """Range metadata per attention kind, once per forward (shared by all layers, heads, fwd and bwd)."""
        if self.N > 0 and encoder:
            self.m_enc = ops.attn_ranges(self.B, self.N, self.N, self.enc_lo, self.enc_hi, device=dev)
        if self.M > 0:
            self.m_dec = ops.attn_ranges(self.B, self.M, self.M, self.dec_lo, self.dec_hi, device=dev)
            self.m_x = ops.attn_ranges(self.B, self.M, self.N, self.x_lo, self.x_hi, device=dev)
        self.p_enc = self.p_dec = self.p_x = None
        if ops.KernelTimer.active is not None:   # mask-aware (query, key) pair counts for the timing breakdown (device scalars)
            cnt = lambda lo, hi: None if lo is None else (hi.long() - lo.long()).clamp(min=0).sum()
            self.p_enc, self.p_dec, self.p_x = cnt(self.enc_lo, self.enc_hi), cnt(self.dec_lo, self.dec_hi), cnt(self.x_lo, self.x_hi)


def _check_epoch(ref, seen):
    """The bf16 operand buffers are re-cast IN PLACE after every optimizer step (EgoM2P._refresh_operands); a backward that
    runs after such a refresh of a forward made before it would silently use the new weights in its dgrad GEMMs. The
    reference raises a saved-tensor version error in that situation; so does this."""
    if ref[0] != seen:
        raise RuntimeError("egom2p_b200: the bf16 weight operands saved by this forward were refreshed (weights changed and "
                           "another forward ran) before its backward; run backward before the next forward of updated weights")


def _zeros(n, dev):
    return torch.zeros(n, dtype=f32, device=dev)


# Bumped by every backward of the block / context / head functions below. The bf16 operand cache of EgoM2P is keyed on it:
# weights whose gradients were just produced are about to be rewritten by an optimizer, and the fused CUDA optimizers
# (torch._fused_adamw_) do not bump Tensor._version, so the version counter alone would leave the cache stale.
_GRAD_GEN = ops.GRAD_GEN


def _split_w13_grad(dw13, F):
    """dw13 rows are interleaved [32 x fc1 | 32 x fc3] groups (see EgoM2P._bf16_w13): back to (fc1.grad, fc3.grad)."""
    Fp, D = dw13.shape[0] // 2, dw13.shape[1]
    v = dw13.view(Fp // 32, 2, 32, D)
    return v[:, 0].reshape(Fp, D)[:F], v[:, 1].reshape(Fp, D)[:F]


def _with_bf16(dx, dxb):
    """Hands the bf16 copy of a residual-stream gradient (written by the LayerNorm backward that produced it, for 1/3 of the
    traffic of a separate cast pass) to the next backward node: autograd passes the same tensor object on, attributes included."""
    dx._egom2p_bf16 = (dxb, dx._version, dx.data_ptr())
    return dx


def _bf16_of(dx):
    hit = getattr(dx, "_egom2p_bf16", None)
    if hit is not None:
        dxb, ver, ptr = hit
        # an in-place accumulation into dx (a second consumer of the residual stream, a hook) bumps its version: the copy is
        # stale then and is rebuilt from the fp32 gradient
        if ver == dx._version and ptr == dx.data_ptr() and dxb.shape == dx.shape and dxb.device == dx.device and dxb.dtype == bf16:
            return dxb
    return ops.cast_bf16(dx)


def _mlp_fwd(mlp, x1, n2w, n2b, w, params, eps):
    """x1 + mlp(norm2 x1). w: the MLP's bf16 operands (mlp.operands), params: its parameters (mlp.params)."""
    h2, _, mean2, rstd2 = ops.layernorm_fwd(x1, n2w, eps, bias=n2b)
    x2, sm = mlp.fwd(h2, x1, w, params)
    return x2, (mean2, rstd2, h2, *sm)


def _mlp_bwd(mlp, dx2, x1, n2w, w, saved, need):
    """need: whether norm2's weight and bias, then each of mlp.params(), want a gradient (False for an absent bias).
    Returns dx1 (incl. the residual path), its bf16 copy, dn2w, dn2b and the gradients of mlp.params(), None where not
    wanted."""
    mean2, rstd2, h2, *sm = saved
    dh2, dparams = mlp.bwd(_bf16_of(dx2), h2, w, sm, need[2:])
    dn2w = _zeros(n2w.numel(), dx2.device) if need[0] else None
    dn2b = _zeros(n2w.numel(), dx2.device) if need[1] else None
    dx1, dx1b = ops.layernorm_bwd(dh2, x1, n2w, mean2, rstd2, dx_in=dx2, d_weight=dn2w, want_bf16=True, d_bias=dn2b)
    return dx1, dx1b, dn2w, dn2b, dparams


def _self_attn_fwd(x, n1w, wqkv, wproj, B, L, H, meta, eps, pairs, bias):
    """bias: the (norm1, qkv, proj) biases, fp32 or None each."""
    D = x.shape[-1]
    n1b, bqkv, bproj = bias
    h1, _, mean1, rstd1 = ops.layernorm_fwd(x, n1w, eps, bias=n1b)
    qkv = ops.linear_fwd(h1, wqkv, bias=bqkv)
    o, lse = ops.attn_fwd(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], B, H, L, L, meta=meta, pairs=pairs)
    x1 = ops.linear_fwd(o, wproj, bias=bproj, addend=x, out_dtype=f32)
    return x1, (mean1, rstd1, h1, qkv, o, lse)


def _self_attn_bwd(dx1, dx1b, x, n1w, wqkv, wproj, saved, B, L, H, meta, pairs, need):
    """need: whether the weight and bias of norm1, qkv and proj want a gradient (False for an absent bias). Returns dx,
    dn1w, dn1b, dwqkv, dbqkv, dwproj, dbproj, None for each gradient not wanted."""
    mean1, rstd1, h1, qkv, o, lse = saved
    D = x.shape[-1]
    need_n1w, need_n1b, need_wqkv, need_bqkv, need_wproj, need_bproj = need
    dwproj = ops.linear_wgrad(dx1b, o) if need_wproj else None
    do = ops.linear_dgrad(dx1b, wproj)
    dqkv = torch.empty_like(qkv)
    ops.attn_bwd(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], o, do, lse, B, H, L, L, dqkv[:, :D], dqkv[:, D:2 * D],
                 dqkv[:, 2 * D:], meta=meta, pairs=pairs)
    dwqkv = ops.linear_wgrad(dqkv, h1) if need_wqkv else None
    dh1 = ops.linear_dgrad(dqkv, wqkv)
    dn1w = _zeros(n1w.numel(), x.device) if need_n1w else None
    dn1b = _zeros(n1w.numel(), x.device) if need_n1b else None
    dbqkv = ops.colsum_bf16(dqkv) if need_bqkv else None
    dbproj = ops.colsum_bf16(dx1b) if need_bproj else None
    dx, dxb = ops.layernorm_bwd(dh1, x, n1w, mean1, rstd1, dx_in=dx1, d_weight=dn1w, want_bf16=True, d_bias=dn1b)
    return _with_bf16(dx, dxb), dn1w, dn1b, dwqkv, dbqkv, dwproj, dbproj


def _cross_fwd(y1, context, qnw, cnw, wq, wkv, wxproj, g, bias):
    """y2 = y1 + cross_attn(query_norm y1, context_norm context). bias: the (query_norm, context_norm, q, kv, proj) biases,
    fp32 or None each."""
    D = y1.shape[-1]
    qnb, cnb, bq, bkv, bxproj = bias
    hq, _, meanq, rstdq = ops.layernorm_fwd(y1, qnw, g.eps, bias=qnb)
    q = ops.linear_fwd(hq, wq, bias=bq)
    hc, _, meanc, rstdc = ops.layernorm_fwd(context, cnw, g.eps, bias=cnb)
    kv = ops.linear_fwd(hc, wkv, bias=bkv)
    o2, lse2 = ops.attn_fwd(q, kv[:, :D], kv[:, D:], g.B, g.H, g.M, g.N, meta=g.m_x, pairs=g.p_x)
    y2 = ops.linear_fwd(o2, wxproj, bias=bxproj, addend=y1, out_dtype=f32)
    return y2, (meanq, rstdq, hq, q, meanc, rstdc, hc, kv, o2, lse2)


def _cross_bwd(g, ctx_key, dy2, dy2b, y1, context, qnw, cnw, wq, wkv, wxproj, saved, need, need_ctx):
    """Backward of _cross_fwd. need: whether the weight and bias of query_norm, context_norm, q, kv and proj want a gradient
    (False for an absent bias); need_ctx: whether `context` does. Returns dy1, dy1b, dctx (None unless this block returns
    the summed context gradient), then dqnw, dqnb, dcnw, dcnb, dwq, dbq, dwkv, dbkv, dwxproj, dbxproj, None for each
    gradient not wanted."""
    meanq, rstdq, hq, q, meanc, rstdc, hc, kv, o2, lse2 = saved
    D = y1.shape[-1]
    dev = y1.device
    need_qnw, need_qnb, need_cnw, need_cnb, need_wq, need_bq, need_wkv, need_bkv, need_wxproj, need_bxproj = need
    # the context side (kv dgrad, context_norm backward) runs for the context's gradient or for context_norm's own
    ctx_side = need_ctx or need_cnw or need_cnb
    dwxproj = ops.linear_wgrad(dy2b, o2) if need_wxproj else None
    do2 = ops.linear_dgrad(dy2b, wxproj)
    dq = torch.empty_like(q)
    dkv = torch.empty_like(kv)
    ops.attn_bwd(q, kv[:, :D], kv[:, D:], o2, do2, lse2, g.B, g.H, g.M, g.N, dq, dkv[:, :D], dkv[:, D:], meta=g.m_x, pairs=g.p_x)
    dwq = ops.linear_wgrad(dq, hq) if need_wq else None
    dhq = ops.linear_dgrad(dq, wq)
    dwkv = ops.linear_wgrad(dkv, hc) if need_wkv else None
    dhc = ops.linear_dgrad(dkv, wkv) if ctx_side else None
    dqnw = _zeros(D, dev) if need_qnw else None
    dcnw = _zeros(D, dev) if need_cnw else None
    dqnb = _zeros(D, dev) if need_qnb else None
    dcnb = _zeros(D, dev) if need_cnb else None
    dbq = ops.colsum_bf16(dq) if need_bq else None
    dbkv = ops.colsum_bf16(dkv) if need_bkv else None
    dbxproj = ops.colsum_bf16(dy2b) if need_bxproj else None
    dy1, dy1b = ops.layernorm_bwd(dhq, y1, qnw, meanq, rstdq, dx_in=dy2, d_weight=dqnw, want_bf16=True, d_bias=dqnb)
    if not need_ctx:
        if ctx_side:   # only context_norm's parameter reductions are wanted; its dx is discarded
            ops.layernorm_bwd(dhc, context, cnw, meanc, rstdc, d_weight=dcnw, d_bias=dcnb)
        return dy1, dy1b, None, dqnw, dqnb, dcnw, dcnb, dwq, dbq, dwkv, dbkv, dwxproj, dbxproj
    # All decoder blocks read the same `context`: instead of letting autograd add twelve (B*N, D) fp32 gradients pairwise,
    # each block's context_norm backward adds the running sum in its own pass (dx_in) and only the block that runs last
    # returns it. g.ctx_users counts the blocks whose forward saw a context that wants a gradient (_DecoderBlockFn.forward).
    # Falls back to one gradient per block whenever the bookkeeping does not match a plain single backward.
    acc = g.dctx_acc
    chained = g.ctx_users > 0 and (acc is None or (acc[0] == ctx_key and acc[1].shape == context.shape))
    last = chained and g.ctx_users == 1
    dctx, dctxb = ops.layernorm_bwd(dhc, context, cnw, meanc, rstdc, dx_in=acc[1] if (chained and acc is not None) else None,
                                    d_weight=dcnw, want_bf16=last, d_bias=dcnb)
    if chained:
        g.ctx_users -= 1
        if last:
            g.dctx_acc = None
            dctx = _with_bf16(dctx, dctxb)
        else:
            g.dctx_acc = (ctx_key, dctx)
            dctx = None
    return dy1, dy1b, dctx, dqnw, dqnb, dcnw, dcnb, dwq, dbq, dwkv, dbkv, dwxproj, dbxproj


class _EncoderBlockFn(torch.autograd.Function):
    """x + attn(norm1 x) then + mlp(norm2 .) -- egom2p_utils.py:356-359. Parameters: weight and bias of norm1, qkv, proj and
    norm2, then mlp.params(); an absent bias is None. The backward computes the gradient of a parameter only when it
    requires one (ctx.needs_input_grad): a frozen parameter gets None and no work is launched for it. dx is always computed."""

    @staticmethod
    def forward(ctx, x, mlp, wb, geom, n1w, n1b, qkv_w, qkv_b, proj_w, proj_b, n2w, n2b, *mlp_params):
        wqkv, wproj, *wm = wb
        g = geom
        x1, sa = _self_attn_fwd(x, n1w, wqkv, wproj, g.B, g.N, g.H, g.m_enc, g.eps, g.p_enc, (n1b, qkv_b, proj_b))
        x2, sm = _mlp_fwd(mlp, x1, n2w, n2b, wm, mlp_params, g.eps)
        ctx.geom, ctx.wb, ctx.mlp = geom, wb, mlp
        ctx.op_epoch = geom.epoch_ref[0]
        ctx.save_for_backward(x, n1w, n2w, x1, *sa, *sm)
        return x2

    @staticmethod
    def backward(ctx, dx2):
        _GRAD_GEN[0] += 1
        _check_epoch(ctx.geom.epoch_ref, ctx.op_epoch)
        x, n1w, n2w, x1, *rest = ctx.saved_tensors
        sa, sm = rest[:6], rest[6:]
        wqkv, wproj, *wm = ctx.wb
        g = ctx.geom
        need = ctx.needs_input_grad
        dx1, dx1b, dn2w, dn2b, dmlp = _mlp_bwd(ctx.mlp, dx2.contiguous(), x1, n2w, wm, sm, need[10:])
        dx, *dsa = _self_attn_bwd(dx1, dx1b, x, n1w, wqkv, wproj, sa, g.B, g.N, g.H, g.m_enc, g.p_enc, need[4:10])
        return (dx, None, None, None, *dsa, dn2w, dn2b, *dmlp)


class _DecoderBlockFn(torch.autograd.Function):
    """self-attn -> cross-attn(query_norm y, context_norm ctx) -> mlp -- egom2p_utils.py:387-391. Parameters: weight and bias
    of norm1, qkv, self-attention proj, query_norm, context_norm, q, kv, cross-attention proj and norm2, then
    mlp.params(); an absent bias is None. As in _EncoderBlockFn, only the parameters that require a gradient get one. dy is
    always computed; the context's gradient (kv dgrad + context_norm backward) only when `context` requires one."""

    @staticmethod
    def forward(ctx, y, context, mlp, wb, geom, n1w, n1b, qkv_w, qkv_b, sproj_w, sproj_b, qnw, qnb, cnw, cnb, q_w, q_b, kv_w,
                kv_b, xproj_w, xproj_b, n2w, n2b, *mlp_params):
        wqkv, wsproj, wq, wkv, wxproj, *wm = wb
        g = geom
        y1, sa = _self_attn_fwd(y, n1w, wqkv, wsproj, g.B, g.M, g.H, g.m_dec, g.eps, g.p_dec, (n1b, qkv_b, sproj_b))
        y2, sx = _cross_fwd(y1, context, qnw, cnw, wq, wkv, wxproj, g, (qnb, cnb, q_b, kv_b, xproj_b))
        y3, sm = _mlp_fwd(mlp, y2, n2w, n2b, wm, mlp_params, g.eps)
        ctx.geom, ctx.wb, ctx.mlp = geom, wb, mlp
        ctx.op_epoch = geom.epoch_ref[0]
        ctx.ctx_key = context.data_ptr()
        if ctx.needs_input_grad[1]:   # this block's backward adds to the summed context gradient (_cross_bwd)
            g.ctx_users += 1
        ctx.save_for_backward(y, context, n1w, qnw, cnw, n2w, y1, y2, *sx, *sa, *sm)
        return y3

    @staticmethod
    def backward(ctx, dy3):
        _GRAD_GEN[0] += 1
        _check_epoch(ctx.geom.epoch_ref, ctx.op_epoch)
        (y, context, n1w, qnw, cnw, n2w, y1, y2, *rest) = ctx.saved_tensors
        sx, sa, sm = rest[:10], rest[10:16], rest[16:]
        wqkv, wsproj, wq, wkv, wxproj, *wm = ctx.wb
        g = ctx.geom
        need = ctx.needs_input_grad
        dy2, dy2b, dn2w, dn2b, dmlp = _mlp_bwd(ctx.mlp, dy3.contiguous(), y2, n2w, wm, sm, need[21:])
        dy1, dy1b, dctx, *dxa = _cross_bwd(g, ctx.ctx_key, dy2, dy2b, y1, context, qnw, cnw, wq, wkv, wxproj, sx, need[11:21],
                                           need[1])
        dy, *dsa = _self_attn_bwd(dy1, dy1b, y, n1w, wqkv, wsproj, sa, g.B, g.M, g.H, g.m_dec, g.p_dec, need[5:11])
        return (dy, dctx, None, None, None, *dsa, *dxa, dn2w, dn2b, *dmlp)


class _ContextFn(torch.autograd.Function):
    """context = decoder_proj_context(encoder_norm(x)) + encoder_emb -- egom2p_model.py:499,722. norm_b: encoder_norm's
    bias (GELU / bias family) or None. The backward skips the projection's dw / db when frozen, and the dgrad and
    encoder_norm backward when neither x nor encoder_norm wants a gradient."""

    @staticmethod
    def forward(ctx, x, enc_emb, norm_w, norm_b, proj_w, proj_b, wb, eps, epoch_ref):
        h, _, mean, rstd = ops.layernorm_fwd(x, norm_w, eps, bias=norm_b)
        context = ops.linear_fwd(h, wb, bias=proj_b, addend=enc_emb, out_dtype=f32)
        ctx.wb = wb
        ctx.epoch_ref, ctx.op_epoch = epoch_ref, epoch_ref[0]
        ctx.save_for_backward(x, norm_w, mean, rstd, h)
        return context

    @staticmethod
    def backward(ctx, dctx):
        _GRAD_GEN[0] += 1
        _check_epoch(ctx.epoch_ref, ctx.op_epoch)
        x, norm_w, mean, rstd, h = ctx.saved_tensors
        need_x, need_emb, need_nw, need_nb, need_pw, need_pb = ctx.needs_input_grad[:6]
        upstream = need_x or need_nw or need_nb
        dctx = dctx.contiguous()
        dcb = _bf16_of(dctx) if (need_pw or upstream) else None
        dw = ops.linear_wgrad(dcb, h) if need_pw else None
        db = ops.colsum(dctx, _zeros(dctx.shape[1], dctx.device)) if need_pb else None
        dx = dnw = dnb = None
        if upstream:
            dh = ops.linear_dgrad(dcb, ctx.wb)
            dnw = _zeros(norm_w.numel(), x.device) if need_nw else None
            dnb = _zeros(norm_w.numel(), x.device) if need_nb else None
            dx, dxb = ops.layernorm_bwd(dh, x, norm_w, mean, rstd, d_weight=dnw, want_bf16=need_x, d_bias=dnb)
            dx = _with_bf16(dx, dxb) if need_x else None
        return dx, dctx if need_emb else None, dnw, dnb, dw, db, None, None, None


class _EmbedFn(torch.autograd.Function):
    """Fused token-embedding + pos/mod-embedding + masked gather for one side (north-star kernel 1).
    args: n token tables (encoder) or the mask token (decoder), then n modality embeddings."""

    @staticmethod
    def forward(ctx, plan, meta, is_decoder, *params):
        lens, vocabs, ids, pos, dim = meta
        n = len(lens)
        if is_decoder:
            mask_token, mods = params[0], params[1:]
            x0, emb = ops.embed_gather_fwd(plan, dim, lens, vocabs, None, None, pos, [m.reshape(-1) for m in mods],
                                           mask_token=mask_token.reshape(-1), want_emb=False)
        else:
            tables, mods = params[:n], params[n:]
            x0, emb = ops.embed_gather_fwd(plan, dim, lens, vocabs, ids, list(tables), pos, [m.reshape(-1) for m in mods])
        ctx.plan, ctx.meta, ctx.is_decoder = plan, meta, is_decoder
        ctx.shapes = [p.shape for p in params]
        ctx.save_for_backward(*[m for m in mods])
        R = plan.rows if plan.rows is not None else plan.B * plan.budget
        if is_decoder:
            return x0.reshape(R, dim)
        return x0.reshape(R, dim), emb.reshape(R, dim)

    @staticmethod
    def backward(ctx, dx0, demb=None):
        lens, vocabs, ids, pos, dim = ctx.meta
        n = len(lens)
        mods = ctx.saved_tensors
        dev = dx0.device
        dx0 = dx0.contiguous()
        # a frozen table, mask token or modality embedding gets no gradient buffer: the kernel skips null outputs
        need = ctx.needs_input_grad[3:]
        d_mods = [_zeros(dim, dev) if nd else None for nd in need[len(need) - n:]]
        if ctx.is_decoder:
            d_tok = _zeros(dim, dev) if need[0] else None
            ops.embed_gather_bwd(ctx.plan, dim, lens, vocabs, None, pos, [m.reshape(-1) for m in mods], dx0, None, None,
                                 d_mods, d_tok)
            grads = [d_tok] + d_mods
        else:
            d_tabs = [torch.zeros(s, dtype=f32, device=dev) if nd else None for s, nd in zip(ctx.shapes[:n], need[:n])]
            ops.embed_gather_bwd(ctx.plan, dim, lens, vocabs, ids, pos, [m.reshape(-1) for m in mods], dx0,
                                 demb.contiguous() if demb is not None else None, d_tabs, d_mods, None)
            grads = d_tabs + d_mods
        return (None, None, None, *[None if g is None else g.reshape(s) for g, s in zip(grads, ctx.shapes)])


class _HeadLossFn(torch.autograd.Function):
    """decoder_norm -> per-modality vocabulary head -> cross-entropy (egom2p_model.py:523,614-680) with the head GEMM
    fused into the softmax statistics: logits live in TMEM only. Returns the per-modality mean CE (0 for empty). The
    backward skips the dW GEMM of a frozen head, and the dY GEMMs, the scatter and the decoder_norm backward when neither
    y nor decoder_norm wants a gradient."""
    CHUNK = 8192

    @staticmethod
    def forward(ctx, y, norm_w, norm_b, rows, targets, wbs, eps, epoch_ref, *head_w):
        ctx.epoch_ref, ctx.op_epoch = epoch_ref, epoch_ref[0]
        yn, _, mean, rstd = ops.layernorm_fwd(y, norm_w, eps, bias=norm_b)
        losses, lses, yms = [], [], []
        for idx, tgt, wb in zip(rows, targets, wbs):
            if idx.numel() == 0:
                losses.append(torch.zeros((), dtype=f32, device=y.device))
                lses.append(None); yms.append(None)
                continue
            ym = ops.gather_rows_bf16(yn, idx)
            loss_sum, lse = ops.ce_forward(ym, wb, tgt)
            losses.append(loss_sum[0] / idx.numel())
            lses.append(lse); yms.append(ym)
        ctx.rows, ctx.targets, ctx.wbs, ctx.lses, ctx.yms = rows, targets, wbs, lses, yms
        ctx.save_for_backward(y, norm_w, mean, rstd)
        return tuple(losses)

    @staticmethod
    def backward(ctx, *dlosses):
        _GRAD_GEN[0] += 1
        _check_epoch(ctx.epoch_ref, ctx.op_epoch)
        y, norm_w, mean, rstd = ctx.saved_tensors
        dev = y.device
        D = y.shape[1]
        need_y, need_nw, need_nb = ctx.needs_input_grad[:3]
        need_heads = ctx.needs_input_grad[8:]
        want_dyn = need_y or need_nw or need_nb   # the dY GEMMs, the scatter and the decoder_norm backward
        dyn = torch.zeros_like(y) if want_dyn else None  # rows of pads / modalities without targets get zero gradient
        dws = []
        for idx, tgt, wb, lse, ym, dl, need_w in zip(ctx.rows, ctx.targets, ctx.wbs, ctx.lses, ctx.yms, dlosses, need_heads):
            V = wb.shape[0]
            if idx.numel() == 0 or dl is None or not (need_w or want_dyn):
                dws.append(torch.zeros(V, D, dtype=f32, device=dev) if need_w else None)
                continue
            R = idx.numel()
            gscale = (dl.reshape(1).to(f32) / R).contiguous()
            dw = torch.empty(V, D, dtype=f32, device=dev) if need_w else None
            dym = torch.empty(R, D, dtype=f32, device=dev) if want_dyn else None
            chunk = min(V, _HeadLossFn.CHUNK)
            buf = torch.empty(R, chunk, dtype=bf16, device=dev)
            for v0 in range(0, V, chunk):
                vc = min(chunk, V - v0)
                dlog = buf[:, :vc]
                ops.ce_dlogits(ym, wb, tgt, lse, gscale, v0, vc, dlog)
                if want_dyn:
                    ops.gemm(dlog, wb[v0:v0 + vc], R, D, vc, b_mn=True, addend=dym if v0 else None, out_f32=dym)
                if need_w:   # a frozen (tied) head gets no dW GEMM
                    ops.gemm(dlog, ym, vc, D, R, a_mn=True, b_mn=True, out_f32=dw[v0:v0 + vc])
            if want_dyn:
                ops.scatter_rows_f32(dym, idx, dyn)
            dws.append(dw)
        dy = dnw = dnb = None
        if want_dyn:
            dnw = _zeros(D, dev) if need_nw else None
            dnb = _zeros(D, dev) if need_nb else None
            dy, dyb = ops.layernorm_bwd(dyn, y, norm_w, mean, rstd, d_weight=dnw, want_bf16=need_y, d_bias=dnb)
            dy = _with_bf16(dy, dyb) if need_y else None
        return (dy, dnw, dnb, None, None, None, None, None, *dws)


# =============================================================================================== the module
class EgoM2P(nn.Module):
    """B200-native EgoM2P. Same constructor arguments as the reference (egom2p_model.py:84-108)."""

    def __init__(self,
                 encoder_embeddings: Dict[str, nn.Module],
                 decoder_embeddings: Dict[str, nn.Module],
                 modality_info: Dict[str, Any],
                 dim: int = 768,
                 encoder_depth: int = 12,
                 decoder_depth: int = 12,
                 num_heads: int = 12,
                 mlp_ratio: float = 4.0,
                 qkv_bias: bool = True,
                 proj_bias: bool = True,
                 mlp_bias: bool = True,
                 drop_path_rate_encoder: float = 0.0,
                 drop_path_rate_decoder: float = 0.0,
                 shared_drop_path: bool = False,
                 act_layer: nn.Module = nn.GELU,
                 norm_layer: Union[partial, nn.Module] = partial(LayerNorm, eps=1e-6, bias=False),
                 gated_mlp: bool = False,
                 qk_norm: bool = False,
                 decoder_causal_mask: bool = False,
                 decoder_sep_mask: bool = True,
                 num_register_tokens: int = 0,
                 use_act_checkpoint: bool = False,
                 share_modality_embeddings: bool = True):
        super().__init__()
        swiglu = not (qkv_bias or proj_bias or mlp_bias) and gated_mlp and act_layer is nn.SiLU
        gelu = qkv_bias and proj_bias and mlp_bias and not gated_mlp and act_layer is nn.GELU
        if qk_norm or not (swiglu or gelu):
            raise NotImplementedError("egom2p_b200 implements the swiglu / no-bias family (egom2p_*_swiglu_nobias) and the "
                                      "GELU / bias family (egom2p_*_gelu)")
        if drop_path_rate_encoder or drop_path_rate_decoder:
            raise NotImplementedError("drop_path > 0 is not built (the reference trains ego-b with 0)")
        if num_register_tokens:
            raise NotImplementedError("register tokens are not built (default 0 in the reference CLI)")
        if dim % num_heads or dim // num_heads != 64:
            raise NotImplementedError("attention kernels are specialised for head_dim 64 (tiny/small/base variants)")
        self.modality_info = modality_info
        self.dim, self.num_heads = dim, num_heads
        self.decoder_causal_mask, self.decoder_sep_mask = decoder_causal_mask, decoder_sep_mask
        self.init_std = 0.02
        self.use_act_checkpoint = use_act_checkpoint
        self.num_register_tokens = num_register_tokens
        eps_probe = norm_layer(4)
        if gelu and not isinstance(getattr(eps_probe, "bias", None), nn.Parameter):
            raise NotImplementedError("the GELU / bias family is built with LayerNorms that have a learnable bias (nn.LayerNorm)")
        self.eps = float(getattr(eps_probe, "eps", 1e-6))
        self.gelu = bool(gelu)
        norm = partial(LayerNorm, eps=self.eps, bias=self.gelu)  # same names/buffers as the reference's LayerNorm

        self.encoder_modalities = set(encoder_embeddings.keys())
        for emb in encoder_embeddings.values():
            emb.init(dim_tokens=dim, init_std=self.init_std)
        self.encoder_embeddings = nn.ModuleDict(encoder_embeddings)
        self.decoder_modalities = set(decoder_embeddings.keys())
        for emb in decoder_embeddings.values():
            emb.init(dim_tokens=dim, init_std=self.init_std)
        self.decoder_embeddings = nn.ModuleDict(decoder_embeddings)
        for side in (self.encoder_embeddings, self.decoder_embeddings):
            for mod, emb in side.items():
                if isinstance(getattr(emb, "pos_emb", None), nn.Parameter):
                    # the fused embed backward emits gradients for the token tables, mask token and modality embeddings only
                    raise NotImplementedError(f"egom2p_b200: adapter '{mod}' has a learnable pos_emb (sincos_pos_emb=False); "
                                              "the fused path supports the fixed sin-cos tables ego-b uses")
        if share_modality_embeddings:
            self.share_modality_embeddings()

        self.encoder = nn.ModuleList([Block(dim, num_heads, mlp_ratio, norm, self.gelu) for _ in range(encoder_depth)])
        self.encoder_norm = norm(dim)
        self.decoder_proj_context = _Linear(dim, dim)
        self.decoder = nn.ModuleList([DecoderBlock(dim, num_heads, mlp_ratio, norm, self.gelu) for _ in range(decoder_depth)])
        self.decoder_norm = norm(dim)
        self.mask_token = nn.Parameter(torch.zeros(1, 1, dim))
        nn.init.normal_(self.mask_token, std=self.init_std)
        self.register_tokens = None
        self.init_weights()
        self._wcache: Dict[Any, tuple] = {}
        self._wplan = None
        self._epoch = [0]   # bumped by every in-place refresh of the bf16 operands (see _check_epoch)
        self.static_target_rows: Optional[Dict[str, int]] = None   # {modality: valid target rows in the batch}, see forward
        self.fixed_decoder_order: Optional[List[str]] = None
        self._static_rows_dev = None
        self.pack_rows = True   # ragged batches: run every per-row kernel over the valid tokens only (see forward)

    # ------------------------------------------------------------------ construction helpers (reference :179-249)
    def share_modality_embeddings(self):
        for mod in self.encoder_modalities & self.decoder_modalities:
            self.decoder_embeddings[mod].mod_emb = self.encoder_embeddings[mod].mod_emb

    def init_weights(self):
        for name, m in self.named_modules():
            if "tokenizer" in name:
                continue
            if isinstance(m, nn.Linear):
                if "qkv" in name:
                    val = math.sqrt(6. / float(m.weight.shape[0] // 3 + m.weight.shape[1]))
                    nn.init.uniform_(m.weight, -val, val)
                elif "kv" in name:
                    val = math.sqrt(6. / float(m.weight.shape[0] // 2 + m.weight.shape[1]))
                    nn.init.uniform_(m.weight, -val, val)
                else:
                    nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, (nn.LayerNorm, LayerNorm)) or type(m).__name__ == "LayerNorm":
                nn.init.constant_(m.weight, 1.0)
                if getattr(m, "bias", None) is not None and isinstance(m.bias, nn.Parameter):
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.Embedding):
                nn.init.normal_(m.weight, std=self.init_std)

    def get_num_layers_encoder(self):
        return len(self.encoder)

    def get_num_layers_decoder(self):
        return len(self.decoder)

    def get_num_layers(self):
        return self.get_num_layers_encoder() + self.get_num_layers_decoder()

    @torch.jit.ignore
    def no_weight_decay(self):
        no_wd = set()
        for side, embs in (("encoder_embeddings", self.encoder_embeddings), ("decoder_embeddings", self.decoder_embeddings)):
            for mod, emb in embs.items():
                if hasattr(emb, "no_weight_decay"):
                    no_wd |= {f"{side}.{mod}.{n}" for n in emb.no_weight_decay()}
        return no_wd

    # ------------------------------------------------------------------ bf16 operand cache (refreshed when a master changes)
    def _bf16(self, key, *params: torch.Tensor, pad32: bool = False) -> torch.Tensor:
        """bf16 GEMM operand of one weight (or of the fc1 | fc3 pair). Entries: (ptrs, versions, generation, operand, params)."""
        ptrs = tuple(p.data_ptr() for p in params)
        vers = tuple(p._version for p in params)
        hit = self._wcache.get(key)
        if hit is not None and hit[0] == ptrs:
            if hit[1] == vers and hit[2] == _GRAD_GEN[0]:
                return hit[3]
            self._refresh_operands()   # some master changed: one launch re-casts every registered operand
            hit = self._wcache[key]
            if hit[1] == vers and hit[2] == _GRAD_GEN[0]:
                return hit[3]
        dev = params[0].device
        if len(params) == 1:
            p = params[0]
            pad = (-p.shape[1]) % (32 if pad32 else 8)
            if pad == 0:
                wb = ops.cast_bf16(p.detach())
            else:  # inner dim padded with zero columns so TMA row pitches stay 16-byte multiples (e.g. hidden 682)
                wb = torch.zeros(p.shape[0], p.shape[1] + pad, dtype=bf16, device=dev)
                wb[:, :p.shape[1]].copy_(ops.cast_bf16(p.detach()))
        else:  # fc1 | fc3 -> one N = 2*hidden GEMM operand with rows interleaved in groups of 32 (hidden padded to 32)
            F, D = params[0].shape
            Fp = (F + 31) // 32 * 32
            wb = torch.zeros(2 * Fp, D, dtype=bf16, device=dev)
            v = wb.view(Fp // 32, 2, 32, D)
            for i, p in enumerate(params):
                tmp = ops.cast_bf16(p.detach())
                if Fp != F:
                    tmp = torch.cat([tmp, torch.zeros(Fp - F, D, dtype=bf16, device=dev)], 0)
                v[:, i].copy_(tmp.view(Fp // 32, 32, D))
        self._wcache[key] = (ptrs, vers, _GRAD_GEN[0], wb, params)
        self._wplan = None
        return wb

    def _refresh_operands(self):
        """Re-cast every cached operand whose masters still live at the same addresses, in one launch (ops.CastPlan)."""
        live = {k: e for k, e in self._wcache.items()
                if e[0] == tuple(p.data_ptr() for p in e[4]) and all(p.dim() == 2 and p.is_contiguous() for p in e[4])}
        if not live:
            return
        sig = tuple((k, e[0], e[3].data_ptr()) for k, e in live.items())
        if self._wplan is None or self._wplan[0] != sig:
            items = []
            for e in live.values():
                if len(e[4]) == 1:
                    items.append((e[4][0].detach(), e[3], 0, 0))
                else:
                    items += [(p.detach(), e[3], 32, i) for i, p in enumerate(e[4])]
            self._wplan = (sig, ops.CastPlan(items))
        self._wplan[1].run()
        self._epoch[0] += 1
        for k, e in live.items():
            self._wcache[k] = (e[0], tuple(p._version for p in e[4]), _GRAD_GEN[0], e[3], e[4])

    def invalidate_weight_cache(self):
        """Force a re-cast of every bf16 operand at the next forward. Needed only after an in-place weight update that
        neither bumps Tensor._version nor follows a backward of this module (see _GRAD_GEN)."""
        _GRAD_GEN[0] += 1

    def _enc_weights(self, i: int):
        b = self.encoder[i]
        return (self._bf16(("e", i, "qkv"), b.attn.qkv.weight), self._bf16(("e", i, "proj"), b.attn.proj.weight),
                *b.mlp.operands(self._bf16, ("e", i)))

    def _dec_weights(self, i: int):
        b = self.decoder[i]
        return (self._bf16(("d", i, "qkv"), b.self_attn.qkv.weight), self._bf16(("d", i, "sproj"), b.self_attn.proj.weight),
                self._bf16(("d", i, "q"), b.cross_attn.q.weight), self._bf16(("d", i, "kv"), b.cross_attn.kv.weight),
                self._bf16(("d", i, "xproj"), b.cross_attn.proj.weight), *b.mlp.operands(self._bf16, ("d", i)))

    # ------------------------------------------------------------------ block application (training)
    def _enc_block(self, i, blk, h, g):
        return _EncoderBlockFn.apply(h, blk.mlp, self._enc_weights(i), g,
                                     *_weights_and_biases(blk.norm1, blk.attn.qkv, blk.attn.proj, blk.norm2), *blk.mlp.params())

    def _dec_block(self, i, blk, h, c, g):
        sa, xa = blk.self_attn, blk.cross_attn
        return _DecoderBlockFn.apply(h, c, blk.mlp, self._dec_weights(i), g,
                                     *_weights_and_biases(blk.norm1, sa.qkv, sa.proj, blk.query_norm, blk.context_norm, xa.q,
                                                          xa.kv, xa.proj, blk.norm2), *blk.mlp.params())

    # ------------------------------------------------------------------ blocks without autograd (generation / sampler paths)
    def _self_attn_infer(self, attn, norm, h, wqkv, wproj, B, L, meta):
        return _self_attn_fwd(h, norm.weight, wqkv, wproj, B, L, self.num_heads, meta, self.eps, None,
                              (_bias(norm), _bias(attn.qkv), _bias(attn.proj)))[0]

    def _mlp_infer(self, blk, h, wm):
        return _mlp_fwd(blk.mlp, h, blk.norm2.weight, _bias(blk.norm2), wm, blk.mlp.params(), self.eps)[0]

    def _decoder_infer(self, h, c, g):
        """The decoder blocks over h (g.B * g.M rows, fp32). c: the context rows that g.m_x ranges over, or None when no
        sample has context: a softmax over zero keys times an empty V is exactly 0 (SURVEY.md A5), so each cross-attention
        then adds only its projection's bias, if it has one."""
        B, M, D = g.B, g.M, g.D
        zero = None
        for i, blk in enumerate(self.decoder):
            wqkv, wsproj, wq, wkv, wxproj, *wm = self._dec_weights(i)
            h = self._self_attn_infer(blk.self_attn, blk.norm1, h, wqkv, wsproj, B, M, g.m_dec)
            xa = blk.cross_attn
            if c is not None:
                hq, _, _, _ = ops.layernorm_fwd(h, blk.query_norm.weight, g.eps, save_stats=False, bias=_bias(blk.query_norm))
                q = ops.linear_fwd(hq, wq, bias=_bias(xa.q))
                hc, _, _, _ = ops.layernorm_fwd(c, blk.context_norm.weight, g.eps, save_stats=False, bias=_bias(blk.context_norm))
                kv = ops.linear_fwd(hc, wkv, bias=_bias(xa.kv))
                o2, _ = ops.attn_fwd(q, kv[:, :D], kv[:, D:], B, g.H, M, g.N, meta=g.m_x, want_lse=False)
                h = ops.linear_fwd(o2, wxproj, bias=_bias(xa.proj), addend=h, out_dtype=f32)
            elif _bias(xa.proj) is not None:
                if zero is None:
                    zero = torch.zeros(B * M, D, dtype=bf16, device=h.device)
                h = ops.linear_fwd(zero, wxproj, bias=_bias(xa.proj), addend=h, out_dtype=f32)
            h = self._mlp_infer(blk, h, wm)
        return h

    # ------------------------------------------------------------------ sampler-facing pieces (reference :251-283,483-551)
    def cat_encoder_tensors(self, mod_dict):
        xs, es, ms, mm = [], [], [], []
        for mod, d in mod_dict.items():
            xs.append(d["x"]); es.append(d["emb"]); ms.append(d["input_mask"])
            mm.append(torch.full_like(d["input_mask"], self.modality_info[mod]["id"], dtype=torch.int16))
        return torch.cat(xs, dim=1), torch.cat(es, dim=1), torch.cat(ms, dim=1), torch.cat(mm, dim=1)

    @staticmethod
    def _prefix_ranges(mask: Optional[torch.Tensor], B: int, rows: int, keys: int, dev):
        """(B,1,keys) / (B,keys) key-padding mask or (B,rows,keys) mask (bool, True = masked) -> per-row [lo, hi) key
        ranges, int32 (B, rows). The masks this path meets are one contiguous run per row (SURVEY.md A3). The reduction
        runs on the mask's OWN shape (a key-padding mask costs O(B * keys), not O(B * rows * keys)) and nothing is read
        back: a non-contiguous row trips a device-side assertion (torch._assert_async) instead of a host sync."""
        if mask is None:
            return None, None
        m = mask.to(dev)
        if m.dim() == 2:
            m = m[:, None, :]
        if m.dtype != torch.bool:
            m = m != 0
        if m.shape[0] != B:
            m = m.expand(B, *m.shape[1:])
        r = m.shape[1]                     # 1 for a key-padding mask
        valid = (~m).to(torch.uint8)       # (B, r, keys), one byte per entry
        cnt = valid.sum(-1, dtype=torch.int32)
        first = valid.argmax(-1).to(torch.int32)                      # first valid key (0 when the row has none)
        last = keys - valid.flip(-1).argmax(-1).to(torch.int32)       # one past the last valid key
        torch._assert_async(((last - first == cnt) | (cnt == 0)).all(),
                            "egom2p_b200 attention supports one contiguous key range per query row")
        zero = torch.zeros_like(cnt)
        lo = torch.where(cnt > 0, first, zero)
        hi = torch.where(cnt > 0, last, zero)
        if r != rows:
            lo, hi = lo.expand(B, rows), hi.expand(B, rows)
        return lo.contiguous(), hi.contiguous()

    def forward_encoder(self, x: torch.Tensor, encoder_mask: torch.Tensor) -> torch.Tensor:
        B, N, D = x.shape
        if N == 0:
            return x
        g = self._geom(B, N, 0)
        g.enc_lo, g.enc_hi = self._prefix_ranges(encoder_mask, B, N, N, x.device)
        g.build_meta(x.device)
        h = x.reshape(B * N, D).float().contiguous()
        for i, blk in enumerate(self.encoder):
            h = self._enc_block(i, blk, h, g)
        return self.encoder_norm(h).reshape(B, N, D)

    def forward_decoder(self, y, context, encoder_mask, decoder_attention_mask):
        B, M, D = y.shape
        N = context.shape[1]
        g = self._geom(B, N, M)
        g.x_lo, g.x_hi = self._prefix_ranges(encoder_mask, B, M, N, y.device) if N > 0 else (None, None)
        g.dec_lo, g.dec_hi = self._prefix_ranges(decoder_attention_mask, B, M, M, y.device)
        g.build_meta(y.device, encoder=False)  # no encoder self-attention on this path
        h = y.reshape(B * M, D).float().contiguous()
        if N == 0:
            # Unconditional branch of guided ROAR decoding (generate.py:793-802): no context token at all. Inference only.
            if torch.is_grad_enabled() and (y.requires_grad or any(p.requires_grad for p in self.decoder.parameters())):
                raise NotImplementedError("decoder with an empty context is an inference-only path (wrap it in torch.no_grad())")
            h = self._decoder_infer(h, None, g)
        else:
            c = context.reshape(B * N, D).float().contiguous()
            for i, blk in enumerate(self.decoder):
                h = self._dec_block(i, blk, h, c, g)
        return self.decoder_norm(h).reshape(B, M, D)

    def forward_logits(self, y, decoder_mod_dict, decoder_mod_mask, return_all_logits: bool = False):
        out = {}
        for mod in decoder_mod_dict:
            idx = self.modality_info[mod]["id"]
            rows = y if return_all_logits else y[decoder_mod_mask == idx]
            out[mod] = self.decoder_embeddings[mod].forward_logits(rows)
        return out

    # ------------------------------------------------------------------ generation path (egom2p_b200/generate.py)
    @torch.no_grad()
    def encode_tokens(self, mod_dict, masks: Dict[str, torch.Tensor], budget: int):
        """Encoder half of one generation pass (reference: GenerationSampler.forward_mask_encoder_generation + forward_encoder
        + decoder_proj_context, generate.py:407-444,749-757) straight from token ids: index plan over `masks` (the
        modalities' input masks, possibly emptied for the unconditional branch), fused embed / gather of the `budget` kept
        slots, the encoder blocks and the context projection. Returns (context (B, budget, D) fp32, n_valid (B,) int32);
        no (B, L, D) embedding of the full modalities, no argsort, no host sync."""
        enc_mods = [m for m in mod_dict if m in self.encoder_embeddings]
        first = mod_dict[enc_mods[0]]["tensor"]
        B, dev, D = first.shape[0], first.device, self.dim
        ep = ops.index_plan([masks[m] for m in enc_mods], [self.modality_info[m]["id"] for m in enc_mods], budget)
        N = ep.budget
        lens, vocabs, ids, pos = self._tables("enc", enc_mods, mod_dict, B, dev)
        x, emb = ops.embed_gather_fwd(ep, D, lens, vocabs, ids, [self.encoder_embeddings[m].token_emb.weight.detach() for m in enc_mods],
                                      pos, [self.encoder_embeddings[m].mod_emb.detach().reshape(-1) for m in enc_mods])
        x, emb = x.reshape(B * N, D), emb.reshape(B * N, D)
        g = self._geom(B, N, 0)
        g.enc_lo = torch.zeros(B, N, dtype=torch.int32, device=dev)
        g.enc_hi = ep.n_valid[:, None].expand(B, N).contiguous()
        g.build_meta(dev)
        for i, blk in enumerate(self.encoder):
            wqkv, wproj, *wm = self._enc_weights(i)
            x = self._self_attn_infer(blk.attn, blk.norm1, x, wqkv, wproj, B, N, g.m_enc)
            x = self._mlp_infer(blk, x, wm)
        h, _, _, _ = ops.layernorm_fwd(x, self.encoder_norm.weight.detach(), self.eps, save_stats=False,
                                       bias=_det(_bias(self.encoder_norm)))
        context = ops.linear_fwd(h, self._bf16("ctx", self.decoder_proj_context.weight), bias=self.decoder_proj_context.bias.detach(),
                                 addend=emb, out_dtype=f32)
        return context.reshape(B, N, D), ep.n_valid

    @torch.no_grad()
    def decode_tokens(self, y0: torch.Tensor, context: Optional[torch.Tensor], n_ctx: Optional[torch.Tensor]):
        """Decoder half of one generation pass (generate.py:758-763 with decoder_attention_mask=None): y0 (B, k, D) fp32 decoder
        inputs, context (B, N, D) fp32 with the first n_ctx[b] rows of sample b valid (a sample with n_ctx = 0 has NO context:
        its cross-attention contributes exactly 0, SURVEY A5 (i) -- that is what lets the conditional and the unconditional
        branch of guided decoding share one batch). Returns decoder_norm(y) as (B * k, D) fp32."""
        B, M, D = y0.shape
        dev = y0.device
        N = 0 if context is None else context.shape[1]
        g = self._geom(B, N, M)
        c = None
        if N > 0:
            g.x_lo = torch.zeros(B, M, dtype=torch.int32, device=dev)
            g.x_hi = n_ctx.to(torch.int32)[:, None].expand(B, M).contiguous()
            g.m_x = ops.attn_ranges(B, M, N, g.x_lo, g.x_hi, device=dev, empty_zero=True)
            c = context.reshape(B * N, D)
        g.m_dec = ops.attn_ranges(B, M, M, device=dev)
        return self.decoder_norm(self._decoder_infer(y0.reshape(B * M, D).float().contiguous(), c, g))

    def head_operand(self, mod: str) -> torch.Tensor:
        """Cached bf16 operand of a modality's vocabulary head (V, D)."""
        return self._bf16(("head", mod), self.decoder_embeddings[mod].to_logits.weight)

    @staticmethod
    def _pack_plan(pl: "ops.Plan", n_valid: List[int], budget: int):
        """Packed view of an index plan: the valid slots only (a prefix of every sample's slots), sample after sample.
        Returns (plan over the packed rows, row offset of every sample, valid rows of every sample) -- device tensors built
        from the host counts, no further synchronisation."""
        dev = pl.keep_mod.device
        B = pl.B
        lens = torch.tensor(n_valid, dtype=torch.int32, device=dev)
        off = torch.cumsum(lens, 0, dtype=torch.int32) - lens
        R = int(sum(n_valid))
        ar = torch.arange(R, dtype=torch.int32, device=dev)
        b_of = torch.searchsorted((off + lens).contiguous(), ar, right=True).to(torch.int32)
        slot = (b_of.long() * budget + (ar - off[b_of.long()]).long())          # flat (b, s) index of every packed row
        pp = ops.Plan()
        pp.B, pp.budget, pp.rows, pp.row_batch = B, budget, R, b_of.contiguous()
        pp.keep_mod = pl.keep_mod.reshape(-1)[slot].contiguous()
        pp.keep_pos = pl.keep_pos.reshape(-1)[slot].contiguous()
        pp.pad = torch.zeros(R, dtype=torch.bool, device=dev)
        pp.mod_mask = pl.mod_mask.reshape(-1)[slot]
        pp.n_valid = pl.n_valid
        pp.keep_idx = None
        pp.target_ids = pp.key_lo = pp.key_hi = None
        if pl.target_ids is not None:
            pp.target_ids = pl.target_ids          # indexed by SLOT (the head row lists are slot lists before remapping)
            pp.key_lo = pl.key_lo.reshape(-1)[slot]
            pp.key_hi = pl.key_hi.reshape(-1)[slot]
        pp.slot_index = slot
        pp.slot_to_row = torch.full((B * budget,), -1, dtype=torch.int64, device=dev)
        pp.slot_to_row[slot] = torch.arange(R, dtype=torch.int64, device=dev)
        return pp, off, lens

    def _geom(self, B, N, M) -> _Geom:
        g = _Geom()
        g.B, g.N, g.M, g.H, g.D, g.eps = B, N, M, self.num_heads, self.dim, self.eps
        g.enc_lo = g.enc_hi = g.dec_lo = g.dec_hi = g.x_lo = g.x_hi = None
        g.m_enc = g.m_dec = g.m_x = None
        g.ctx_users, g.dctx_acc = 0, None   # decoder blocks of this forward that read `context` / their running gradient
        g.epoch_ref = self._epoch
        return g

    # ------------------------------------------------------------------ the training step (reference :683-734)
    def _tables(self, side: str, mods: List[str], mod_dict, B, dev):
        embs = self.encoder_embeddings if side == "enc" else self.decoder_embeddings
        lens, vocabs, ids, pos = [], [], [], []
        for m in mods:
            e = embs[m]
            t = mod_dict[m]["tensor"].reshape(B, -1)
            if t.dtype != torch.int64:
                t = t.to(torch.int64)
            ids.append(t.contiguous())
            lens.append(t.shape[1])
            vocabs.append(int(e.vocab_size))
            pos.append(e.pos_emb.detach().reshape(-1, self.dim))
        return lens, vocabs, ids, pos

    def forward(self, mod_dict: Dict[str, Dict[str, torch.Tensor]], num_encoder_tokens: int, num_decoder_tokens: int,
                loss_type: str = "mod", return_logits: bool = False):
        if loss_type not in ("mod", "modality", "weighted_mod", "token"):
            raise ValueError("Invalid loss type")
        enc_mods = [m for m in mod_dict if m in self.encoder_embeddings]
        dec_mods = [m for m in mod_dict if m in self.decoder_embeddings]
        first = mod_dict[enc_mods[0]]["tensor"]
        if not first.is_cuda:
            raise RuntimeError("egom2p_b200: mod_dict tensors must live on a CUDA device (no CPU path exists)")
        B, dev, D = first.shape[0], first.device, self.dim
        ids_of = lambda m: self.modality_info[m]["id"]

        # ---- index plans (no embedding rows touched; masks -> slots, pads, key ranges)
        ep = ops.index_plan([mod_dict[m]["input_mask"] for m in enc_mods], [ids_of(m) for m in enc_mods], num_encoder_tokens)
        # decoder modality order is shuffled exactly like the reference (random.sample over the dict items, :312)
        dec_order = [m for m, _ in random.sample([(m, None) for m in dec_mods], len(dec_mods))]
        if self.fixed_decoder_order is not None:   # CUDA-graph replay: the order drawn at capture time (the loss is order-invariant, A7)
            dec_order = [m for m in self.fixed_decoder_order if m in dec_mods]
        for m in dec_order:
            if self.modality_info[m]["type"] in ("seq", "seq_emb", "seq_token"):
                raise NotImplementedError("sequence (teacher-forced) decoder modalities are not part of the mod4 path")
        dlens, dvocabs, dids, dpos = self._tables("dec", dec_order, mod_dict, B, dev)
        dp = ops.index_plan([mod_dict[m]["target_mask"] for m in dec_order], [ids_of(m) for m in dec_order], num_decoder_tokens,
                            decoder=True, attn_cnt=[mod_dict[m]["decoder_attention_mask"].to(torch.int32) for m in dec_order],
                            ids=dids, causal=self.decoder_causal_mask, sep=self.decoder_sep_mask)
        N, M = ep.budget, dp.budget
        # ---- row lists of the heads, and ONE device -> host copy per forward: valid tokens per sample on both sides and the
        # rows per head (the reference's boolean row-selects sync once per modality, egom2p_model.py:633). With
        # `static_target_rows` set (CUDA-graph capture, egom2p_b200/graphed.py) nothing is copied.
        row_tab, counts = ops.plan_rows(dp.mod_mask, [ids_of(m) for m in dec_mods])
        pack = None
        if self.static_target_rows is not None:
            n_rows = [int(self.static_target_rows[m]) for m in dec_mods]
            key = (tuple(n_rows), dev)
            if self._static_rows_dev is None or self._static_rows_dev[0] != key:   # built outside graph capture (warm-up)
                self._static_rows_dev = (key, torch.tensor(n_rows, dtype=torch.int32, device=dev))
            torch._assert_async((counts == self._static_rows_dev[1]).all(),
                                "egom2p_b200: static_target_rows does not match this batch")
        else:
            host = torch.cat([ep.n_valid, dp.n_valid, counts]).tolist()
            ne, nd, n_rows = host[:B], host[B:2 * B], host[2 * B:]
            # Ragged batch: PACK the rows (valid slots only, sample after sample) so that LayerNorm, every GEMM and the
            # attention queries run over the valid tokens instead of the full budgets (the reference's masks leave ~48 % of
            # the 2048 + 2048 slots valid on average, SURVEY.md section 8(d)). A sample without any encoder token keeps the
            # slot layout: its cross-attention must average over its own pad keys (SURVEY A5 (ii)).
            if self.pack_rows and min(ne) > 0 and (sum(ne) < B * N or sum(nd) < B * M) and sum(nd) > 0:
                pack = (ne, nd)
        if pack is not None:
            ep_p, e_off, e_len = self._pack_plan(ep, pack[0], N)
            dp_p, d_off, d_len = self._pack_plan(dp, pack[1], M)
            Re, Rd = ep_p.rows, dp_p.rows
            g = self._geom(1, Re, Rd)        # one virtual sample: block-diagonal key ranges keep the samples apart
            eb, db = ep_p.row_batch.long(), dp_p.row_batch.long()
            g.enc_lo = e_off[eb].reshape(1, Re).contiguous()
            g.enc_hi = (e_off[eb] + e_len[eb]).reshape(1, Re).contiguous()
            g.x_lo = e_off[db].reshape(1, Rd).contiguous()
            g.x_hi = (e_off[db] + e_len[db]).reshape(1, Rd).contiguous()
            g.dec_lo = (dp_p.key_lo + d_off[db]).reshape(1, Rd).contiguous()
            g.dec_hi = (dp_p.key_hi + d_off[db]).reshape(1, Rd).contiguous()
            ep, dp = ep_p, dp_p
        else:
            g = self._geom(B, N, M)
            nv = ep.n_valid
            g.enc_lo = torch.zeros(B, N, dtype=torch.int32, device=dev)
            g.enc_hi = nv[:, None].expand(B, N).contiguous()
            g.x_lo = torch.zeros(B, M, dtype=torch.int32, device=dev)
            g.x_hi = nv[:, None].expand(B, M).contiguous()
            g.dec_lo, g.dec_hi = dp.key_lo, dp.key_hi
        g.build_meta(dev)

        # ---- fused embed / gather
        elens, evocabs, eids, epos = self._tables("enc", enc_mods, mod_dict, B, dev)
        x, enc_emb = _EmbedFn.apply(ep, (elens, evocabs, eids, epos, D), False,
                                    *[self.encoder_embeddings[m].token_emb.weight for m in enc_mods],
                                    *[self.encoder_embeddings[m].mod_emb for m in enc_mods])
        y = _EmbedFn.apply(dp, (dlens, dvocabs, None, dpos, D), True, self.mask_token,
                           *[self.decoder_embeddings[m].mod_emb for m in dec_order])

        # ---- encoder
        for i, blk in enumerate(self.encoder):
            x = self._enc_block(i, blk, x, g)
        context = _ContextFn.apply(x, enc_emb, self.encoder_norm.weight, _bias(self.encoder_norm), self.decoder_proj_context.weight,
                                   self.decoder_proj_context.bias, self._bf16("ctx", self.decoder_proj_context.weight), self.eps,
                                   self._epoch)
        # ---- decoder
        for i, blk in enumerate(self.decoder):
            y = self._dec_block(i, blk, y, context, g)

        if return_logits:
            yn = self.decoder_norm(y)
            if pack is not None:   # back to the (B, M) slot layout the reference returns (pad slots: zeros)
                full = torch.zeros(B * M, D, dtype=yn.dtype, device=dev)
                full[dp.slot_index] = yn
                yn = full
            yn = yn.reshape(B, M, D)
            return {m: self.decoder_embeddings[m].forward_logits(yn) for m in dec_mods}

        # ---- heads + loss (row lists from plan_rows above; in the packed layout the slot indices are remapped)
        tgt_flat = dp.target_ids.reshape(-1)          # indexed by slot in both layouts
        rows, targets, wbs, heads = [], [], [], []
        for i, m in enumerate(dec_mods):
            idx = row_tab[i, :n_rows[i]]              # slots (b * M + s) of this modality's valid targets, ascending
            targets.append(tgt_flat.index_select(0, idx))
            rows.append(dp.slot_to_row.index_select(0, idx) if pack is not None else idx)
            w = self.decoder_embeddings[m].to_logits.weight
            heads.append(w)
            wbs.append(self._bf16(("head", m), w))
        per_mod = _HeadLossFn.apply(y, self.decoder_norm.weight, _bias(self.decoder_norm), rows, targets, wbs,
                                    self.eps, self._epoch, *heads)
        mod_loss = {}
        for m, l in zip(dec_mods, per_mod):
            if loss_type == "weighted_mod" and rows[dec_mods.index(m)].numel():
                l = l / math.log(self.modality_info[m]["vocab_size"]) * 5.545177444479562
            mod_loss[m] = l
        if loss_type == "token":
            counts = {m: rows[i].numel() * int(self.decoder_embeddings[m].vocab_size) for i, m in enumerate(dec_mods)}
            loss = sum(mod_loss[m] * counts[m] for m in dec_mods) / sum(counts.values())
        else:
            loss = sum(mod_loss.values()) / len(mod_loss)
        return loss, mod_loss

    # ------------------------------------------------------------------ freeze helpers (reference :737-819)
    def _set_grad(self, modules, flag):
        for mod in modules:
            for p in mod.parameters():
                p.requires_grad = flag

    def freeze_encoder(self, freeze_embeddings=True):
        self._set_grad([self.encoder, self.encoder_norm] + ([self.encoder_embeddings] if freeze_embeddings else []), False)

    def freeze_encoder_except_specific_embeddings(self, frozen_embedding_domain):
        doms = frozen_embedding_domain.split("-")
        self._set_grad([self.encoder, self.encoder_norm], False)
        for name, p in self.encoder_embeddings.named_parameters():
            if name.split(".")[0] in doms:
                p.requires_grad = False

    def unfreeze_encoder(self, unfreeze_embeddings=True):
        self._set_grad([self.encoder, self.encoder_norm] + ([self.encoder_embeddings] if unfreeze_embeddings else []), True)

    def freeze_decoder(self, freeze_embeddings=True):
        self._set_grad([self.decoder, self.decoder_norm] + ([self.decoder_embeddings] if freeze_embeddings else []), False)

    def freeze_decoder_except_specific_embeddings(self, frozen_embedding_domain):
        doms = frozen_embedding_domain.split("-")
        self._set_grad([self.decoder, self.decoder_norm], False)
        for name, p in self.decoder_embeddings.named_parameters():
            if name.split(".")[0] in doms:
                p.requires_grad = False

    def unfreeze_decoder(self, unfreeze_embeddings=True):
        self._set_grad([self.decoder, self.decoder_norm] + ([self.decoder_embeddings] if unfreeze_embeddings else []), True)

    def freeze_shared_params(self):
        self.freeze_encoder(freeze_embeddings=False)
        self.freeze_decoder(freeze_embeddings=False)

    def freeze_params_except_specific_embeddings(self, frozen_embedding_domain):
        self.freeze_encoder_except_specific_embeddings(frozen_embedding_domain)
        self.freeze_decoder_except_specific_embeddings(frozen_embedding_domain)

    def unfreeze_shared_params(self):
        self.unfreeze_encoder(unfreeze_embeddings=False)
        self.unfreeze_decoder(unfreeze_embeddings=False)

    def unfreeze_all(self):
        self.unfreeze_encoder(unfreeze_embeddings=True)
        self.unfreeze_decoder(unfreeze_embeddings=True)
