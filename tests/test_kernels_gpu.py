"""GPU parity tests of the individual sm_100a kernels, called through the C ABI (egom2p_b200.ops -> ctypes).
Integer / index / gather work is bit-exact against the oracle; floating-point kernels are compared with a plain
torch fp32 evaluation of the same op on the same bf16-rounded inputs (tolerances stated per test)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import egom2p_oracle as orc  # noqa: E402
import synth  # noqa: E402


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from egom2p_b200 import ops as _ops
    return _ops


def dev(t):
    return t.cuda()


# ------------------------------------------------------------------------------------------ index plan
def _plan_case(ops, cfg, md, n_enc, n_dec, dec_order):
    mods = list(cfg["mods"])
    ids = {m: cfg["mods"][m]["id"] for m in mods}
    B = md[mods[0]]["tensor"].shape[0]
    ep = ops.index_plan([dev(md[m]["input_mask"]) for m in mods], [ids[m] for m in mods], n_enc)
    dp = ops.index_plan([dev(md[m]["target_mask"]) for m in dec_order], [ids[m] for m in dec_order], n_dec, decoder=True,
                        attn_cnt=[dev(md[m]["decoder_attention_mask"]) for m in dec_order],
                        ids=[dev(md[m]["tensor"].reshape(B, -1)) for m in dec_order])
    oe = orc.plan_encoder({m: md[m]["input_mask"].numpy() for m in mods}, ids, n_enc)
    od = orc.plan_decoder({m: md[m]["target_mask"].numpy() for m in mods},
                          {m: md[m]["decoder_attention_mask"].numpy() for m in mods},
                          {m: md[m]["tensor"].reshape(B, -1).numpy() for m in mods}, ids, dec_order, n_dec)
    assert np.array_equal(ep.keep_idx.cpu().numpy(), oe["ids_keep"])
    assert np.array_equal(ep.pad.cpu().numpy(), oe["mask"])
    assert np.array_equal(ep.mod_mask.cpu().numpy(), oe["mod_mask"])
    assert np.array_equal(ep.n_valid.cpu().numpy(), (~oe["mask"]).sum(1))
    assert np.array_equal(dp.keep_idx.cpu().numpy(), od["ids_keep"])
    assert np.array_equal(dp.pad.cpu().numpy(), od["mask"])
    assert np.array_equal(dp.mod_mask.cpu().numpy(), od["mod_mask"])
    assert np.array_equal(dp.target_ids.cpu().numpy(), od["target_ids"])
    # key ranges <-> the reference's dense (B, M, M) mask; rows whose range is empty == fully masked rows
    lo, hi = dp.key_lo.cpu().numpy(), dp.key_hi.cpu().numpy()
    M = lo.shape[1]
    j = np.arange(M)[None, None, :]
    dense = ~((j >= lo[:, :, None]) & (j < hi[:, :, None]))
    assert np.array_equal(dense, od["attn_mask"])
    return ep, dp


def test_index_plan_small_ragged(ops):
    cfg = synth.make_cfg(48, 2, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=128, video_thw=(5, 4, 4))
    md = synth.make_batch(cfg, B=4, seed=11,
                          n_in={"tok_cam": [5, 0, 30, 2], "tok_depth": [30, 10, 0, 1], "tok_gaze": [4, 0, 30, 0], "tok_rgb": [25, 40, 4, 0]},
                          n_tgt={"tok_cam": [10, 30, 0, 1], "tok_depth": [20, 0, 40, 0], "tok_gaze": [3, 0, 0, 0], "tok_rgb": [15, 18, 70, 0]})
    _plan_case(ops, cfg, md, 64, 48, ["tok_depth", "tok_gaze", "tok_cam", "tok_rgb"])
    _plan_case(ops, cfg, md, 220, 220, ["tok_rgb", "tok_cam", "tok_gaze", "tok_depth"])  # budget == every position
    _plan_case(ops, cfg, md, 1, 1, ["tok_rgb", "tok_cam", "tok_gaze", "tok_depth"])


def test_index_plan_egob_golden(ops, golden_dir):
    g = np.load(os.path.join(golden_dir, "plan_egob.npz"))
    cfg = synth.make_cfg(12, 1, 0, 0, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=64000)
    n_in = {"tok_cam": [15, 0, 30, 0], "tok_depth": [1009, 694, 0, 30], "tok_gaze": [15, 0, 30, 30], "tok_rgb": [1009, 0, 5120, 0]}
    n_tg = {"tok_cam": [15, 30, 0, 1], "tok_depth": [1009, 0, 2048, 0], "tok_gaze": [15, 0, 0, 0], "tok_rgb": [1009, 2018, 0, 0]}
    md = synth.make_batch(cfg, B=4, seed=31, n_in=n_in, n_tgt=n_tg)
    ep, dp = _plan_case(ops, cfg, md, 2048, 2048, list(g["dec_order"]))
    assert np.array_equal(ep.keep_idx.cpu().numpy(), g["enc_keep"])
    assert np.array_equal(dp.target_ids.cpu().numpy(), g["target_ids"])
    assert np.array_equal(dp.mod_mask.cpu().numpy(), g["dec_mod"])


# ------------------------------------------------------------------------------------------ fused embed / gather
def test_embed_gather_bit_exact_and_grads(ops, golden_dir):
    g = np.load(os.path.join(golden_dir, "small4.npz"))
    cfg = synth.make_cfg(48, 2, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=128, video_thw=(5, 4, 4))
    sd = synth.make_state_dict(cfg, 5)
    md = synth.make_batch(cfg, B=4, seed=11,
                          n_in={"tok_cam": [5, 0, 30, 2], "tok_depth": [30, 10, 0, 1], "tok_gaze": [4, 0, 30, 0], "tok_rgb": [25, 40, 4, 0]},
                          n_tgt={"tok_cam": [10, 30, 0, 1], "tok_depth": [20, 0, 40, 0], "tok_gaze": [3, 0, 0, 0], "tok_rgb": [15, 18, 70, 0]})
    mods = list(cfg["mods"])
    order = list(g["dec_order"])
    B, D = 4, 48
    ep, dp = _plan_case(ops, cfg, md, 64, 48, order)

    def tabs(side, ms):
        return ([cfg["mods"][m]["len"] for m in ms], [cfg["mods"][m]["vocab"] for m in ms],
                [dev(md[m]["tensor"].reshape(B, -1)) for m in ms],
                [dev(sd[f"{side}.{m}.token_emb.weight"]) for m in ms],
                [dev(sd[f"{side}.{m}.pos_emb"][0]).contiguous() for m in ms],
                [dev(sd[f"{side}.{m}.mod_emb"].reshape(-1)) for m in ms])
    lens, vocs, ids, tb, pos, mod = tabs("encoder_embeddings", mods)
    x0, emb = ops.embed_gather_fwd(ep, D, lens, vocs, ids, tb, pos, mod)
    assert np.array_equal(x0.cpu().numpy(), g["enc_x0"])      # bit-exact vs the reference itself
    assert np.array_equal(emb.cpu().numpy(), g["enc_emb"])
    dlens, dvocs, dids, dtb, dpos, dmod = tabs("decoder_embeddings", order)
    y0, _ = ops.embed_gather_fwd(dp, D, dlens, dvocs, None, None, dpos, dmod, mask_token=dev(sd["mask_token"].reshape(-1)), want_emb=False)
    assert np.array_equal(y0.cpu().numpy(), g["dec_y0"])

    # backward: scatter-add into the tables / modality embeddings vs torch autograd on the oracle's gather
    gen = torch.Generator().manual_seed(0)
    dx0 = torch.randn(B, 64, D, generator=gen)
    demb = torch.randn(B, 64, D, generator=gen)
    tb_ref = [sd[f"encoder_embeddings.{m}.token_emb.weight"].clone().requires_grad_() for m in mods]
    mod_ref = [sd[f"encoder_embeddings.{m}.mod_emb"].clone().requires_grad_() for m in mods]
    xs = torch.cat([tb_ref[i][md[m]["tensor"].reshape(B, -1)] for i, m in enumerate(mods)], 1)
    es = torch.cat([(sd[f"encoder_embeddings.{m}.pos_emb"] + mod_ref[i]).expand(B, -1, -1) for i, m in enumerate(mods)], 1)
    keep = torch.from_numpy(orc.plan_encoder({m: md[m]["input_mask"].numpy() for m in mods},
                                             {m: cfg["mods"][m]["id"] for m in mods}, 64)["ids_keep"])[..., None].expand(-1, -1, D)
    pad = torch.from_numpy(g["enc_mask"])[..., None]
    xg = torch.gather(xs, 1, keep).masked_fill(pad, 0.0)
    eg = torch.gather(es, 1, keep).masked_fill(pad, 0.0)
    ((xg + eg) * dx0).sum().backward(retain_graph=True)
    (eg * demb).sum().backward()
    d_tabs = [torch.zeros_like(t).cuda() for t in tb_ref]
    d_mods = [torch.zeros(D).cuda() for _ in mods]
    ops.embed_gather_bwd(ep, D, lens, vocs, ids, pos, mod, dev(dx0), dev(demb), d_tabs, d_mods, None)
    for i in range(len(mods)):
        torch.testing.assert_close(d_tabs[i].cpu(), tb_ref[i].grad, rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(d_mods[i].cpu(), mod_ref[i].grad.reshape(-1), rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------------------------------ layernorm / elementwise
@pytest.mark.parametrize("rows,dim", [(37, 256), (1000, 768), (64, 384), (5, 48), (34751, 768), (1, 768)])
def test_layernorm_fwd_bwd(ops, rows, dim):
    gen = torch.Generator().manual_seed(rows)
    x = torch.randn(rows, dim, generator=gen) * 2 + 0.5
    w = 1 + 0.1 * torch.randn(dim, generator=gen)
    dy = torch.randn(rows, dim, generator=gen)
    res = torch.randn(rows, dim, generator=gen)
    xr, wr = x.clone().requires_grad_(), w.clone().requires_grad_()
    y = torch.nn.functional.layer_norm(xr, (dim,), wr, None, 1e-6)
    y.backward(dy)
    yb, yf, mean, rstd = ops.layernorm_fwd(dev(x), dev(w), out_bf16=True, out_f32=True)
    torch.testing.assert_close(yf.cpu(), y.detach(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(yb.cpu().float(), y.detach(), rtol=1e-2, atol=1e-2)
    dw = torch.zeros(dim, device="cuda")
    dx, dxb = ops.layernorm_bwd(dev(dy), dev(x), dev(w), mean, rstd, dx_in=dev(res), d_weight=dw, want_bf16=True)
    torch.testing.assert_close(dx.cpu(), xr.grad + res, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(dw.cpu(), wr.grad, rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(dxb.cpu().float(), xr.grad + res, rtol=1e-2, atol=2e-2)
    dx2, _ = ops.layernorm_bwd(dev(dy).bfloat16(), dev(x), dev(w), mean, rstd)
    torch.testing.assert_close(dx2.cpu(), xr.grad, rtol=5e-2, atol=2e-2)


def test_cast(ops):
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(1001, generator=gen)
    assert torch.equal(ops.cast_bf16(dev(x)).cpu(), x.bfloat16())


def test_fused_adamw_and_clip_match_torch_per_tensor_steps():
    """Optimizer tail (egom2p/utils/native_scaler.py:27-47): multi-tensor grad-norm + AdamW with the clip folded in, against
    torch.nn.utils.clip_grad_norm_ + torch.optim.AdamW over two parameter groups, odd sizes, 4 steps, a changing lr and a
    parameter without gradient."""
    from egom2p_b200.optim import FusedAdamW, FusedScalerWithGradNormCount
    gen = torch.Generator().manual_seed(3)
    shapes = [(5000,), (33, 7), (1, 1, 768), (8193,), (64, 129), (3,)]
    p_ref = [torch.randn(s, generator=gen).requires_grad_() for s in shapes]
    p_new = [torch.nn.Parameter(dev(p.detach().clone())) for p in p_ref]
    frozen_ref, frozen_new = torch.randn(10).requires_grad_(), torch.nn.Parameter(torch.randn(10, device="cuda"))
    kw = dict(lr=1e-3, betas=(0.9, 0.95), eps=1e-8)
    groups = lambda ps, fr: [{"params": ps[:3] + [fr], "weight_decay": 0.05}, {"params": ps[3:], "weight_decay": 0.0}]
    o_ref = torch.optim.AdamW(groups(p_ref, frozen_ref), **kw)
    o_new = FusedAdamW(groups(p_new, frozen_new), **kw)
    scaler = FusedScalerWithGradNormCount(enabled=False)
    for step in range(4):
        for g_ref, g_new in zip(o_ref.param_groups, o_new.param_groups):
            g_ref["lr"] = g_new["lr"] = 1e-3 * (1 + step)            # the reference scheduler rewrites param_group["lr"] each step
        scale = 50.0 if step % 2 else 0.01                             # norm above and below max_norm = 1
        grads = [torch.randn(s, generator=gen) * scale for s in shapes]
        for p, g in zip(p_ref, grads):
            p.grad = g.clone()
        n_ref = torch.nn.utils.clip_grad_norm_(p_ref + [frozen_ref], 1.0)
        o_ref.step()
        # the same gradients through backward() on the GPU side
        loss = sum((p * dev(g)).sum() for p, g in zip(p_new, grads))
        n_new = scaler(loss, o_new, clip_grad=1.0, parameters=p_new)
        o_new.zero_grad(set_to_none=True)
        torch.testing.assert_close(n_new.cpu(), n_ref, rtol=1e-5, atol=0)
    for a, b in zip(p_new, p_ref):
        torch.testing.assert_close(a.detach().cpu(), b.detach(), rtol=2e-5, atol=2e-6)
    assert [int(o_new.state[p]["step"]) for p in p_new] == [int(o_ref.state[p]["step"]) for p in p_ref] == [4] * len(shapes)
    assert frozen_new.grad is None and not o_new.state[frozen_new]


# ------------------------------------------------------------------------------------------ tcgen05 GEMM
def _ref_mm(a, b):
    return a.double() @ b.double().t()


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (256, 768, 768), (2048, 2304, 768), (1000, 520, 328), (4096, 768, 2048),
                                   (77, 64, 40), (19000, 768, 768)])
def test_gemm_tn(ops, M, N, K):
    gen = torch.Generator().manual_seed(M + N + K)
    a = (torch.randn(M, K, generator=gen)).bfloat16()
    b = (torch.randn(N, K, generator=gen) / K ** 0.5).bfloat16()
    ref = _ref_mm(a, b).float()
    out = torch.empty(M, N, dtype=torch.float32, device="cuda")
    ops.gemm(dev(a), dev(b), M, N, K, out_f32=out)
    torch.testing.assert_close(out.cpu(), ref, rtol=1e-3, atol=1e-3)
    outb = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    ops.gemm(dev(a), dev(b), M, N, K, out_bf16=outb)
    torch.testing.assert_close(outb.cpu().float(), ref, rtol=1e-2, atol=1e-2)


def test_gemm_epilogue_bias_residual_strided(ops):
    M, N, K = 640, 768, 768
    gen = torch.Generator().manual_seed(3)
    big = torch.randn(M, 3 * K, generator=gen).bfloat16()   # A is a column slice of a packed matrix (lda = 3K)
    a = big[:, K:2 * K]
    b = (torch.randn(N, K, generator=gen) / K ** 0.5).bfloat16()
    bias = torch.randn(N, generator=gen)
    res = torch.randn(M, N, generator=gen)
    ref = (_ref_mm(a, b) + bias.double() + res.double()).float()
    bigd = dev(big)
    out = dev(res.clone())
    ops.gemm(bigd[:, K:2 * K], dev(b), M, N, K, bias=dev(bias), addend=out, out_f32=out)   # in-place residual
    torch.testing.assert_close(out.cpu(), ref, rtol=1e-3, atol=2e-3)


@pytest.mark.parametrize("R,N,K", [(512, 768, 2304), (1000, 328, 520), (4096, 2048, 768)])
def test_gemm_dgrad_wgrad_layouts(ops, R, N, K):
    """dgrad: dX = dY W (B consumed MN-major); wgrad: dW = dY^T X (both operands MN-major)."""
    gen = torch.Generator().manual_seed(R)
    dy = torch.randn(R, N, generator=gen).bfloat16()
    w = (torch.randn(N, K, generator=gen) / N ** 0.5).bfloat16()
    x = torch.randn(R, K, generator=gen).bfloat16()
    dx = ops.linear_dgrad(dev(dy), dev(w), out_dtype=torch.float32)
    torch.testing.assert_close(dx.cpu(), (dy.double() @ w.double()).float(), rtol=1e-3, atol=2e-3)
    dw = ops.linear_wgrad(dev(dy), dev(x))
    ref = (dy.double().t() @ x.double()).float()
    torch.testing.assert_close(dw.cpu(), ref, rtol=1e-3, atol=1e-3 * R ** 0.5)
    dw2 = ops.linear_wgrad(dev(dy), dev(x), out=dw, accumulate=True)
    torch.testing.assert_close(dw2.cpu(), 2 * ref, rtol=1e-3, atol=2e-3 * R ** 0.5)


# ------------------------------------------------------------------------------------------ head + CE
@pytest.mark.parametrize("R,V,K", [(300, 256, 256), (1000, 64000, 768), (17, 1000, 384)])
def test_fused_head_cross_entropy(ops, R, V, K):
    gen = torch.Generator().manual_seed(R)
    y = torch.randn(R, K, generator=gen).bfloat16()
    w = (torch.randn(V, K, generator=gen) * 0.05).bfloat16()
    tgt = torch.randint(0, V, (R,), generator=gen)
    logits = (y.double() @ w.double().t())
    ref_lse = torch.logsumexp(logits, -1)
    ref_loss = torch.nn.functional.cross_entropy(logits, tgt, reduction="sum")
    loss, lse = ops.ce_forward(dev(y), dev(w), dev(tgt))
    torch.testing.assert_close(lse.cpu().double(), ref_lse, rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(loss.cpu().double()[0], ref_loss, rtol=1e-5, atol=1e-2)
    # dlogits chunk
    gscale = torch.tensor([0.37], device="cuda")
    v0, vc = (0, V) if V <= 1000 else (32000, 8000)
    dl = torch.empty(R, vc, dtype=torch.bfloat16, device="cuda")
    ops.ce_dlogits(dev(y), dev(w), dev(tgt), lse, gscale, v0, vc, dl)
    p = torch.softmax(logits, -1)
    p[torch.arange(R), tgt] -= 1
    ref = (p * 0.37)[:, v0:v0 + vc].float()
    torch.testing.assert_close(dl.cpu().float(), ref, rtol=2e-2, atol=1e-5)


# ------------------------------------------------------------------------------------------ attention forward
def attn_ranges(B, Mq, Nk, mode):
    """Key ranges [lo, hi) (B, Mq) int32 of the attention tests (shared with tests/test_attention_bwd_gpu.py)."""
    lo = torch.zeros(B, Mq, dtype=torch.int32)
    if mode == "full":
        hi = torch.full((B, Mq), Nk, dtype=torch.int32)
    elif mode == "prefix":   # encoder / cross: keys [0, n_b); one sample has an empty range -> uniform rows
        n = torch.tensor([Nk - 3, 0][:B] if B > 1 else [Nk - 3], dtype=torch.int32)
        hi = n[:, None].expand(B, Mq).contiguous()
    else:                    # decoder self: contiguous modality segments + a pad tail with empty ranges
        assert mode in ("segments", "causal")
        bounds = [0, Mq // 2 - 11, Mq - 40, Mq - 25, Mq - 10]
        hi = torch.zeros(B, Mq, dtype=torch.int32)
        for a, b_ in zip(bounds[:-1], bounds[1:]):
            lo[:, a:b_] = a
            # causal: row i sees [segment start, i + 1) -- a different end on every row
            hi[:, a:b_] = torch.arange(a + 1, b_ + 1, dtype=torch.int32) if mode == "causal" else b_
    return lo, hi


def _attn_ref(q, k, v, lo, hi, H):
    """fp64 reference with the reference's masked_fill(-finfo.max) semantics. q (B,Mq,H*64), k/v (B,Nk,H*64)."""
    B, Mq, _ = q.shape
    Nk = k.shape[1]
    qh = q.double().reshape(B, Mq, H, 64).permute(0, 2, 1, 3)
    kh = k.double().reshape(B, Nk, H, 64).permute(0, 2, 1, 3)
    vh = v.double().reshape(B, Nk, H, 64).permute(0, 2, 1, 3)
    s = qh @ kh.transpose(-1, -2) * 64 ** -0.5
    j = torch.arange(Nk)[None, None, :]
    masked = ~((j >= lo[:, :, None]) & (j < hi[:, :, None]))
    s = s.masked_fill(masked[:, None], -torch.finfo(torch.float32).max)
    p = s.softmax(-1)
    return (p @ vh).permute(0, 2, 1, 3).reshape(B, Mq, H * 64), s


@pytest.mark.parametrize("gain", [1.0, 3.0])   # 1: |q| max|k| scale log2e ~ 15 -> bound-path softmax; 3: ~ 140 -> online-maximum path
@pytest.mark.parametrize("B,H,Mq,Nk,mode", [(2, 3, 200, 200, "prefix"), (1, 2, 128, 64, "full"), (2, 4, 300, 517, "prefix"),
                                            (2, 2, 260, 260, "segments"), (1, 1, 20, 24, "prefix"), (1, 12, 2048, 2048, "segments"),
                                            (2, 2, 256, 384, "prefix"),    # B > 1 with whole tiles: the TMA-store epilogue
                                            (2, 2, 260, 260, "causal"), (1, 3, 700, 700, "causal")])
def test_attention_fwd(ops, B, H, Mq, Nk, mode, gain):
    gen = torch.Generator().manual_seed(Mq * 7 + Nk)
    D = H * 64
    qkv = torch.randn(B, Mq, 3 * D, generator=gen)
    qkv[..., :2 * D] *= gain
    qkv = qkv.bfloat16()
    kvsrc = qkv if Mq == Nk else torch.randn(B, Nk, 3 * D, generator=gen).mul_(torch.tensor([gain] * (2 * D) + [1.0] * D)).bfloat16()
    q, k, v = qkv[..., :D], kvsrc[..., D:2 * D], kvsrc[..., 2 * D:]
    lo, hi = attn_ranges(B, Mq, Nk, mode)
    ref, s_ref = _attn_ref(q, k, v, lo.long(), hi.long(), H)
    qd, kd = dev(qkv).reshape(B * Mq, 3 * D), dev(kvsrc).reshape(B * Nk, 3 * D)
    o, lse = ops.attn_fwd(qd[:, :D], kd[:, D:2 * D], kd[:, 2 * D:], B, H, Mq, Nk, dev(lo), dev(hi))
    torch.testing.assert_close(o.cpu().float().reshape(B, Mq, D), ref.float(), rtol=2e-2, atol=2e-2)
    # saved statistic (consumed by the backward): log2-sum-exp of the scaled scores over the row's range
    rows = (hi > lo)
    lse_ref = torch.logsumexp(s_ref, -1) * 1.4426950408889634       # (B, H, Mq)
    got = lse.cpu()[:, :, :Mq].double()
    for b in range(B):
        torch.testing.assert_close(got[b][:, rows[b]], lse_ref[b][:, rows[b]], rtol=1e-3, atol=2e-2)


def test_attention_fwd_no_keys(ops):
    """Sampler's unconditional pass: zero context tokens -> cross-attention contributes exactly 0 (SURVEY A5 (i))."""
    q = torch.randn(40, 128, generator=torch.Generator().manual_seed(0)).bfloat16().cuda()
    o, _ = ops.attn_fwd(q, q, q, 1, 2, 40, 0)
    assert torch.count_nonzero(o) == 0
