"""GPU: attention backward (prep + dQ + dK/dV kernels) vs torch autograd (fp64) on the same bf16 inputs."""
import pytest
import torch

from test_kernels_gpu import attn_ranges

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available()
    from egom2p_b200 import ops as _ops
    return _ops


def _ref(q, k, v, do, lo, hi, H):
    B, Mq, _ = q.shape
    Nk = k.shape[1]
    q, k, v = (t.double().requires_grad_() for t in (q, k, v))
    qh = q.reshape(B, Mq, H, 64).permute(0, 2, 1, 3)
    kh = k.reshape(B, Nk, H, 64).permute(0, 2, 1, 3)
    vh = v.reshape(B, Nk, H, 64).permute(0, 2, 1, 3)
    s = qh @ kh.transpose(-1, -2) * 64 ** -0.5
    j = torch.arange(Nk)[None, None, :]
    masked = ~((j >= lo[:, :, None]) & (j < hi[:, :, None]))
    s = s.masked_fill(masked[:, None], -torch.finfo(torch.float32).max)
    o = (s.softmax(-1) @ vh).permute(0, 2, 1, 3).reshape(B, Mq, H * 64)
    o.backward(do.double())
    return o.detach(), q.grad, k.grad, v.grad


@pytest.mark.parametrize("gain", [1.0, 3.0])   # 1: |q| max|k| scale log2e ~ 15 -> bound-path softmax; 3: ~ 140 -> online-maximum path
@pytest.mark.parametrize("B,H,Mq,Nk,mode", [(1, 1, 128, 128, "full"), (2, 3, 200, 200, "prefix"), (2, 2, 300, 517, "prefix"),
                                            (2, 2, 260, 260, "segments"), (1, 1, 20, 24, "prefix"), (1, 12, 2048, 2048, "segments"),
                                            (2, 2, 256, 384, "prefix"),    # B > 1 with whole tiles: the TMA-store epilogue
                                            (2, 2, 260, 260, "causal"), (1, 3, 700, 700, "causal")])
def test_attention_bwd(ops, B, H, Mq, Nk, mode, gain):
    gen = torch.Generator().manual_seed(Mq * 5 + Nk)
    D = H * 64
    qkv = torch.randn(B, Mq, 3 * D, generator=gen)
    qkv[..., :2 * D] *= gain
    qkv = qkv.bfloat16()
    kvsrc = qkv if Mq == Nk else torch.randn(B, Nk, 3 * D, generator=gen).mul_(torch.tensor([gain] * (2 * D) + [1.0] * D)).bfloat16()
    do = torch.randn(B, Mq, D, generator=gen).bfloat16()
    q, k, v = qkv[..., :D], kvsrc[..., D:2 * D], kvsrc[..., 2 * D:]
    lo, hi = attn_ranges(B, Mq, Nk, mode)
    o_ref, dq_ref, dk_ref, dv_ref = _ref(q, k, v, do, lo.long(), hi.long(), H)
    qd, kd = qkv.cuda().reshape(B * Mq, 3 * D), kvsrc.cuda().reshape(B * Nk, 3 * D)
    lod, hid = lo.cuda(), hi.cuda()
    o, lse = ops.attn_fwd(qd[:, :D], kd[:, D:2 * D], kd[:, 2 * D:], B, H, Mq, Nk, lod, hid)
    dqkv = torch.zeros(B * Mq, 3 * D, dtype=torch.bfloat16, device="cuda")
    if Mq == Nk:
        dq, dk, dv = dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:]     # packed gradient, written in place
    else:
        dq = dqkv[:, :D]
        dkv = torch.zeros(B * Nk, 2 * D, dtype=torch.bfloat16, device="cuda")
        dk, dv = dkv[:, :D], dkv[:, D:]
    ops.attn_bwd(qd[:, :D], kd[:, D:2 * D], kd[:, 2 * D:], o, do.cuda().reshape(B * Mq, D), lse, B, H, Mq, Nk, dq, dk, dv, lod, hid)
    torch.testing.assert_close(o.cpu().float().reshape(B, Mq, D), o_ref.float(), rtol=2e-2, atol=2e-2)
    for name, got, ref in (("dq", dq, dq_ref), ("dk", dk, dk_ref), ("dv", dv, dv_ref)):
        got = got.float().cpu().reshape(ref.shape)
        err = (got - ref.float()).abs().max().item()
        scale = ref.abs().max().item() + 1e-6
        assert err <= 3e-2 * scale + 1e-3, f"{name}: max err {err} vs scale {scale}"
