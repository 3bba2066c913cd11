"""GPU: the attention and GEMM kernels at the shapes of packed ragged batches (DESIGN.md section 4, "row packing").

A packed batch runs as ONE virtual sample of R = sum(n_valid) rows: the key ranges are block-diagonal, their boundaries fall
anywhere inside the 64- and 128-row blocks of the kernels, and every weight gradient has K = R, a length that is never a
multiple of 64. Every case here compares a kernel with a plain fp64 torch evaluation of the same op on the same bf16 inputs,
run on the device. Packed attention references are computed per sample (one dense attention per query segment and key range,
never an R x R matrix), and every error is checked per sample against that sample's own scale, so that a one-token sample
cannot pass under the scale of a 2048-token neighbour. Tolerances are those of tests/test_kernels_gpu.py,
tests/test_attention_bwd_gpu.py and tests/test_swiglu_gemm_gpu.py."""
import pytest
import torch
import torch.nn.functional as F

from test_swiglu_gemm_gpu import interleave

pytestmark = pytest.mark.gpu

bf16, f64 = torch.bfloat16, torch.float64
LOG2E = 1.4426950408889634
SCALE = 64 ** -0.5
BOUND_LIMIT = 60.0                                   # kBoundLimit in egom2p_b200/csrc/attn.cu
DEC_ORDER = ["tok_rgb", "tok_gaze", "tok_depth", "tok_cam"]
# Sample lengths of the synthetic packing: segment boundaries on both sides of the 64- and 128-row block edges.
SYN_LENS = [1, 63, 64, 65, 127, 128, 129, 2048, 5]


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from egom2p_b200 import ops as _ops
    return _ops


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(gen, *shape):
    return torch.randn(*shape, device="cuda", generator=gen)


# ------------------------------------------------------------------------------------------------ packed plans
def _packed_ranges(ops, b, offset, causal=False):
    """Packs a batch of reference-distribution masks (tests/test_ragged_masks_gpu.py) the way EgoM2P.forward does and returns
    its key ranges over the virtual sample: {"enc" | "x" | "dec": (lo, hi)} as (R,) int32, plus the row offsets and lengths
    of every sample on both sides."""
    import bench
    from egom2p_b200.modality_info import MODALITY_INFO
    from egom2p_b200.model import EgoM2P
    md = bench.make_batch_ref_masks(b, offset, 5 + offset, pin=False)
    mods = sorted(md)
    ids = lambda ms: [MODALITY_INFO[m]["id"] for m in ms]
    ep = ops.index_plan([md[m]["input_mask"].cuda() for m in mods], ids(mods), bench.N_ENC)
    dp = ops.index_plan([md[m]["target_mask"].cuda() for m in DEC_ORDER], ids(DEC_ORDER), bench.N_DEC, decoder=True,
                        attn_cnt=[md[m]["decoder_attention_mask"].cuda() for m in DEC_ORDER],
                        ids=[md[m]["tensor"].reshape(b, -1).cuda() for m in DEC_ORDER], causal=causal)
    ne, nd = ep.n_valid.tolist(), dp.n_valid.tolist()
    assert min(ne) > 0 and min(nd) > 0
    ep_p, e_off, e_len = EgoM2P._pack_plan(ep, ne, ep.budget)
    dp_p, d_off, d_len = EgoM2P._pack_plan(dp, nd, dp.budget)
    eb, db = ep_p.row_batch.long(), dp_p.row_batch.long()
    # exactly as egom2p_b200/model.py:1095-1100 derives the packed ranges
    r = {"enc": (e_off[eb], e_off[eb] + e_len[eb]),
         "x": (e_off[db], e_off[db] + e_len[db]),
         "dec": (dp_p.key_lo + d_off[db], dp_p.key_hi + d_off[db])}
    r = {k: (lo.int().contiguous(), hi.int().contiguous()) for k, (lo, hi) in r.items()}
    r.update(e_off=e_off.tolist(), e_len=ne, d_off=d_off.tolist(), d_len=nd)
    return r


@pytest.fixture(scope="module")
def real_plan(ops):
    """32 samples of the reference-distribution masks: ~35 k encoder and ~28 k decoder rows."""
    return _packed_ranges(ops, 32, 0)


def _segments(lens):
    off = [0]
    for n in lens:
        off.append(off[-1] + n)
    return [(off[i], off[i + 1]) for i in range(len(lens))]


def _syn_ranges(lens, kind):
    """Synthetic packed ranges over samples of the given lengths: "enc" = the sample's own rows; "dec" = two modality
    segments per sample (split at a third), shifted by the sample offset."""
    lo, hi = [], []
    for a, b in _segments(lens):
        n = b - a
        cuts = [a, b] if kind == "enc" or n < 2 else [a, a + n // 3, b]
        for s0, s1 in zip(cuts[:-1], cuts[1:]):
            lo += [s0] * (s1 - s0)
            hi += [s1] * (s1 - s0)
    t = lambda x: torch.tensor(x, dtype=torch.int32, device="cuda")
    return t(lo), t(hi)


# ------------------------------------------------------------------------------------------------ attention
def _attn_ref(q, k, v, lo, hi, H, do=None):
    """fp64 attention of ONE sample: q (M, H*64), k / v (N, H*64), row i sees keys [lo_i, hi_i) (all non-empty).
    Returns o (M, H*64), lse (H, M) in log2 units, and (dq, dk, dv) when do is given."""
    M, N = q.shape[0], k.shape[0]
    q, k, v = (t.to(f64).requires_grad_(do is not None) for t in (q, k, v))
    qh, kh, vh = (t.reshape(-1, H, 64).transpose(0, 1) for t in (q, k, v))
    j = torch.arange(N, device=q.device)
    keep = (j[None, :] >= lo[:, None].long()) & (j[None, :] < hi[:, None].long())
    s = (qh @ kh.transpose(-1, -2) * SCALE).masked_fill(~keep, float("-inf"))
    o = (s.softmax(-1) @ vh).transpose(0, 1).reshape(M, H * 64)
    lse = torch.logsumexp(s, -1).detach() * LOG2E
    if do is None:
        return o.detach(), lse, None
    o.backward(do.to(f64))
    return o.detach(), lse, (q.grad, k.grad, v.grad)


def _max_err(got, ref):
    return (got.to(f64) - ref).abs().max().item(), ref.abs().max().item()


def _run_packed(ops, H, q, k, v, lo, hi, segs, backward=True, do=None, seed=0):
    """Runs forward (and backward) over the virtual sample (B = 1) and checks every sample against its own fp64 reference.
    q (Mq, H*64), k / v (Nk, H*64) bf16 views; lo / hi (Mq,) int32; segs: the query rows [a, b) of every sample (each
    sample's key span is the union of its rows' ranges). Returns the kernel outputs."""
    Mq, Nk, D = q.shape[0], k.shape[0], H * 64
    lo2, hi2 = lo[None].contiguous(), hi[None].contiguous()
    meta = ops.attn_ranges(1, Mq, Nk, lo2, hi2)
    o, lse = ops.attn_fwd(q, k, v, 1, H, Mq, Nk, meta=meta)
    if backward:
        if do is None:
            do = _randn(_gen(seed + 1), Mq, D).to(bf16)
        dq = torch.zeros(Mq, D, dtype=bf16, device="cuda")
        dk = torch.zeros(Nk, D, dtype=bf16, device="cuda")
        dv = torch.zeros(Nk, D, dtype=bf16, device="cuda")
        ops.attn_bwd(q, k, v, o, do, lse, 1, H, Mq, Nk, dq, dk, dv, meta=meta)
    lo_h, hi_h = lo.tolist(), hi.tolist()
    for i, (a, b) in enumerate(segs):
        ka, kb = min(lo_h[a:b]), max(hi_h[a:b])
        assert kb > ka
        o_ref, lse_ref, grads = _attn_ref(q[a:b], k[ka:kb], v[ka:kb], lo[a:b] - ka, hi[a:b] - ka, H,
                                          do[a:b] if backward else None)
        err, scale = _max_err(o[a:b], o_ref)
        assert err <= 2e-2 * scale, f"sample {i} rows [{a}, {b}): o max err {err} vs scale {scale}"
        torch.testing.assert_close(lse[0, :, a:b].to(f64), lse_ref, rtol=1e-3, atol=2e-2, msg=lambda m: f"sample {i} lse: {m}")
        if backward:
            for name, got, ref in (("dq", dq[a:b], grads[0]), ("dk", dk[ka:kb], grads[1]), ("dv", dv[ka:kb], grads[2])):
                err, scale = _max_err(got, ref)
                assert err <= 3e-2 * scale + 1e-3, f"sample {i} rows [{a}, {b}): {name} max err {err} vs scale {scale}"
    return o, lse


def _qkv(seed, R, H):
    return _randn(_gen(seed), R, 3 * H * 64).to(bf16)


def test_packed_encoder_self_real_plan(ops, real_plan):
    """Case 1: encoder self-attention over the whole virtual sample, B = 1, Mq = Nk = Re, H = 12."""
    lo, hi = real_plan["enc"]
    R, H, D = lo.numel(), 12, 768
    assert R > 20000
    qkv = _qkv(1, R, H)
    segs = [(a, a + n) for a, n in zip(real_plan["e_off"], real_plan["e_len"])]
    _run_packed(ops, H, qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], lo, hi, segs)


def test_packed_decoder_self_real_plan(ops, real_plan):
    """Case 2: decoder self-attention: the modality segments of every sample shifted by its row offset."""
    lo, hi = real_plan["dec"]
    R, H, D = lo.numel(), 12, 768
    qkv = _qkv(2, R, H)
    segs = [(a, a + n) for a, n in zip(real_plan["d_off"], real_plan["d_len"])]
    _run_packed(ops, H, qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], lo, hi, segs)


def test_packed_decoder_causal(ops):
    """Case 2, causal: index_plan(..., causal=1) over a few samples, packed; a different key end on almost every row."""
    r = _packed_ranges(ops, 4, 3, causal=True)
    lo, hi = r["dec"]
    assert (hi[1:] != hi[:-1]).float().mean().item() > 0.9
    R, H, D = lo.numel(), 4, 256
    qkv = _qkv(3, R, H)
    segs = [(a, a + n) for a, n in zip(r["d_off"], r["d_len"])]
    _run_packed(ops, H, qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], lo, hi, segs)


def test_packed_cross_real_plan(ops, real_plan):
    """Case 3: cross-attention, Mq = Rd queries against Nk = Re keys; query and key segments at different offsets."""
    lo, hi = real_plan["x"]
    Rd, Re, H, D = lo.numel(), len(real_plan["enc"][0]), 12, 768
    g = _gen(4)
    q = _randn(g, Rd, D).to(bf16)
    kv = _randn(g, Re, 2 * D).to(bf16)
    segs = [(a, a + n) for a, n in zip(real_plan["d_off"], real_plan["d_len"])]
    _run_packed(ops, H, q, kv[:, :D], kv[:, D:], lo, hi, segs)


@pytest.mark.parametrize("kind", ["enc", "dec"])
def test_packed_self_synthetic(ops, kind):
    """Cases 1 and 2 on the synthetic packing: segment boundaries around every 64- / 128-row block edge."""
    lo, hi = _syn_ranges(SYN_LENS, kind)
    R, H, D = lo.numel(), 2, 128
    qkv = _qkv(5, R, H)
    _run_packed(ops, H, qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], lo, hi, _segments(SYN_LENS))


def test_packed_cross_synthetic(ops):
    """Case 3 on the synthetic packing: a sample with exactly one encoder token, and query segments in another order of
    lengths than the key segments, so that no boundary lines up between the two sides."""
    e_lens = SYN_LENS
    d_lens = [5, 129, 2048, 1, 64, 63, 128, 65, 127]
    e_segs, d_segs = _segments(e_lens), _segments(d_lens)
    lo = torch.cat([torch.full((b - a,), ea, dtype=torch.int32) for (a, b), (ea, _) in zip(d_segs, e_segs)]).cuda()
    hi = torch.cat([torch.full((b - a,), eb, dtype=torch.int32) for (a, b), (_, eb) in zip(d_segs, e_segs)]).cuda()
    H, D = 2, 128
    g = _gen(6)
    q = _randn(g, d_segs[-1][1], D).to(bf16)
    kv = _randn(g, e_segs[-1][1], 2 * D).to(bf16)
    _run_packed(ops, H, q, kv[:, :D], kv[:, D:], lo, hi, d_segs)


def _tile_bound(q, k, H, B=1):
    """m_r = |q_r| max|k| scale log2e per row (max |k| over the whole (batch, head), as the kernel's pre-pass), reduced to
    its maximum per 128-row tile: (H, tiles). A tile takes the online-maximum path when this exceeds kBoundLimit."""
    M = q.shape[0]
    qn = q.to(f64).reshape(M, H, 64).norm(dim=-1)                        # (M, H)
    kn = k.to(f64).reshape(-1, H, 64).norm(dim=-1).max(0).values          # (H,)
    m = (qn * kn * SCALE * LOG2E).t()                                     # (H, M)
    pad = (-M) % 128
    return F.pad(m, (0, pad)).reshape(H, -1, 128).max(-1).values


def test_packed_isolation_mixed_paths(ops):
    """Case 4: one sample with keys x8 and values x1e3 inside the virtual sample. max|k| is taken over the whole virtual
    sample, so its neighbours' tiles either move to the online path (|q| normal) or stay on the bound path with P far
    below 1 (the 2048-row sample, |q| x0.25). Every sample, the large one included, must still match its own reference,
    and so must its dK / dV."""
    lens = SYN_LENS
    segs = _segments(lens)
    lo, hi = _syn_ranges(lens, "enc")
    R, H, D = lo.numel(), 2, 128
    qkv = _randn(_gen(7), R, 3 * D)
    big, quiet = lens.index(129), lens.index(2048)
    a, b = segs[big]
    qkv[a:b, D:2 * D] *= 8
    qkv[a:b, 2 * D:] *= 1e3
    a, b = segs[quiet]
    qkv[a:b, :D] *= 0.25
    qkv = qkv.to(bf16)
    assert torch.isfinite(qkv.float()).all()
    q, k, v = qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:]
    m = _tile_bound(q, k, H)
    assert (m > BOUND_LIMIT).any() and (m < BOUND_LIMIT).any(), m
    _run_packed(ops, H, q, k, v, lo, hi, segs)


@pytest.mark.parametrize("sigma", [0.15, 1.0])
def test_bound_limit_corner(ops, sigma):
    """Case 5: rows with m_r in (50, 60) -- the bound path -- whose true maximum score lies far below the bound: keys
    anti-aligned with the queries (plus noise of scale sigma), values at scale 1e-2. The smallest P = 2^(s - m_r) goes down
    to about 2^-115 (sigma = 1) and 2^-119 (sigma = 0.15), the range attn.cu:16-21 claims to represent exactly.
    The backward runs at sigma = 1 only: at sigma = 0.15 the keys agree to 1 %, dQ = scale * sum_j dS_j (k_j - mean k) cancels
    a component 100 times its result, and rounding dS or O to bf16 alone (the operands of any bf16 backward) moves dQ by
    6 % of its scale in fp64 -- the kernel could not be held to 3e-2 there without a wider tolerance."""
    H, D, M, N = 2, 128, 256, 192
    g = _gen(8)
    u = _randn(g, H, 64)
    u = u / u.norm(dim=-1, keepdim=True)                                  # one query direction per head
    k = (-17.0 * u[None] + sigma * _randn(g, N, H, 64)).reshape(N, D).to(bf16)
    kmax = k.to(f64).reshape(N, H, 64).norm(dim=-1).max(0).values         # (H,)
    target = torch.linspace(50.5, 59.5, M, device="cuda", dtype=f64)      # m_r of every row
    a = target[:, None] / (kmax[None, :] * SCALE * LOG2E)                 # (M, H) query norms
    q = (a[..., None] * u[None].to(f64)).reshape(M, D).to(bf16)
    v = (1e-2 * _randn(g, N, D)).to(bf16)
    qn = q.to(f64).reshape(M, H, 64).norm(dim=-1)
    m_r = qn * kmax[None] * SCALE * LOG2E                                 # (M, H)
    assert m_r.min().item() > 50 and m_r.max().item() < BOUND_LIMIT
    s = torch.einsum("mhd,nhd->mhn", q.to(f64).reshape(M, H, 64), k.to(f64).reshape(N, H, 64)) * SCALE * LOG2E
    assert (s.max(-1).values - m_r).max().item() < -80                    # every row's largest P is below 2^-80
    assert (s.min(-1).values - m_r).min().item() < -114                   # the smallest reach 2^-114 and below
    lo = torch.zeros(M, dtype=torch.int32, device="cuda")
    hi = torch.full((M,), N, dtype=torch.int32, device="cuda")
    do = (100 * _randn(_gen(9), M, D)).to(bf16)                           # gradients of order 1 and above
    _run_packed(ops, H, q, k, v, lo, hi, [(0, M)], backward=sigma >= 1.0, do=do)


@pytest.mark.parametrize("Mq,Nk,lens", [(200, 300, [0, 37, 300]), (10, 9387, [0, 37, 9387])])
def test_empty_zero(ops, Mq, Nk, lens):
    """Case 6: the sampler's batched cond / uncond pass (empty_zero = 1): the rows of the sample without context are exactly 0,
    the other samples match their reference. Nk = 9387 is the largest encoder length of the generation tests."""
    B, H, D = len(lens), 2, 128
    g = _gen(10 + Mq)
    q = _randn(g, B * Mq, D).to(bf16)
    kv = _randn(g, B * Nk, 2 * D).to(bf16)
    n = torch.tensor(lens, dtype=torch.int32, device="cuda")
    lo = torch.zeros(B, Mq, dtype=torch.int32, device="cuda")
    hi = n[:, None].expand(B, Mq).contiguous()
    meta = ops.attn_ranges(B, Mq, Nk, lo, hi, empty_zero=True)
    o, lse = ops.attn_fwd(q, kv[:, :D], kv[:, D:], B, H, Mq, Nk, meta=meta)
    o = o.reshape(B, Mq, D)
    for b, nb in enumerate(lens):
        if nb == 0:
            assert torch.count_nonzero(o[b]) == 0
            continue
        ks = slice(b * Nk, b * Nk + nb)
        o_ref, lse_ref, _ = _attn_ref(q[b * Mq:(b + 1) * Mq], kv[ks, :D], kv[ks, D:], lo[b], hi[b], H)
        err, scale = _max_err(o[b], o_ref)
        assert err <= 2e-2 * scale, f"sample {b}: o max err {err} vs scale {scale}"
        torch.testing.assert_close(lse[b, :, :Mq].to(f64), lse_ref, rtol=1e-3, atol=2e-2)


# ------------------------------------------------------------------------------------------------ GEMM: ragged split-K wgrad
def _split_plan(M, N, K, sms):
    """Python mirror of the fp32-output GEMM's tile width and split-K choice (gemm.cu:721-741, :763-767) for a wgrad (fp32
    output, no bias, no foreign addend). Used only to show that the sweep below reaches every split regime; the kernel
    results are checked against fp64, not against this. Returns (BN, splits, k_blocks)."""
    BM, BK = 128, 64
    BN = 256 if N >= 256 else 128
    k_blocks = (K + BK - 1) // BK
    units = (((M + BM - 1) // BM + 1) // 2) * ((N + BN - 1) // BN)
    workers = sms // 2
    splits = 1
    if units < 3 * workers and k_blocks >= 16:
        best = units / (((units + workers - 1) // workers) * workers)
        if units < workers:
            best = 0.0
        for r in range(1, 5):
            sp = max(min(workers * r // units, k_blocks // 8), 1)
            util = units * sp / (((units * sp + workers - 1) // workers) * workers)
            if util > best + (0.02 if units < workers else 0.10):
                best, splits = util, sp
        kb_per = (k_blocks + splits - 1) // splits
        splits = (k_blocks + kb_per - 1) // kb_per
    return BN, splits, k_blocks


WGRAD_SHAPES = [(2304, 768), (768, 768), (4096, 768), (768, 2048), (256, 768)]
WGRAD_K = [1023, 1024, 1025, 2047, 34751]


def test_wgrad_sweep_covers_split_regimes():
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    plans = {(o, i, K): _split_plan(o, i, K, sms)[1] for o, i in WGRAD_SHAPES for K in WGRAD_K}
    splits = set(plans.values())
    assert 1 in splits and 2 in splits and max(splits) >= 3, plans
    # a ragged K: its partial last k-block lies in the last split of a split-K launch
    assert any(s > 1 and K % 64 for (_, _, K), s in plans.items()), plans


@pytest.mark.parametrize("out_f,in_f", WGRAD_SHAPES)
@pytest.mark.parametrize("K", WGRAD_K)
def test_wgrad_ragged_split_k(ops, out_f, in_f, K):
    """dW = dY^T X with K = R packed rows, plain and accumulated into C (tolerance of test_gemm_dgrad_wgrad_layouts)."""
    g = _gen(K + out_f + in_f)
    dy = _randn(g, K, out_f).to(bf16)
    x = _randn(g, K, in_f).to(bf16)
    ref = dy.to(f64).t() @ x.to(f64)
    dw = ops.linear_wgrad(dy, x)
    torch.testing.assert_close(dw.to(f64), ref, rtol=1e-3, atol=1e-3 * K ** 0.5)
    prev = _randn(g, out_f, in_f) * K ** 0.5
    acc = ops.linear_wgrad(dy, x, out=prev.clone(), accumulate=True)
    torch.testing.assert_close(acc.to(f64), ref + prev.to(f64), rtol=1e-3, atol=2e-3 * K ** 0.5)


# ------------------------------------------------------------------------------------------------ GEMM: epilogues at ragged M
EPI_M = [1, 129, 6949, 34751]


def _check_bf16(got, ref, tol=2e-2):
    err, scale = _max_err(got, ref)
    assert err <= tol * scale, f"max err {err} vs scale {scale}"


@pytest.mark.parametrize("M", EPI_M)
def test_store_epilogues_ragged_rows(ops, M):
    """bf16 output with bias (N = 2304: BN = 256 at M = 34751, BN = 128 at M = 129), the in-place fp32 residual, and the
    bf16 dgrad with B MN-major (both tile widths as well)."""
    g = _gen(M)
    K, N = 768, 2304
    x = _randn(g, M, K).to(bf16)
    w = (_randn(g, N, K) * K ** -0.5).to(bf16)
    bias = _randn(g, N)
    _check_bf16(ops.linear_fwd(x, w, bias=bias), x.to(f64) @ w.to(f64).t() + bias.to(f64))
    # in-place residual (fp32): out = x w^T + bias + out
    w2 = (_randn(g, 768, K) * K ** -0.5).to(bf16)
    b2 = _randn(g, 768)
    res = _randn(g, M, 768)
    out = res.clone()
    ops.gemm(x, w2, M, 768, K, bias=b2, addend=out, out_f32=out)
    torch.testing.assert_close(out.to(f64), x.to(f64) @ w2.to(f64).t() + b2.to(f64) + res.to(f64), rtol=1e-3, atol=2e-3)
    # dgrad dX = dY W (bf16 out), W consumed MN-major
    dy = _randn(g, M, N).to(bf16)
    _check_bf16(ops.linear_dgrad(dy, w), dy.to(f64) @ w.to(f64))


@pytest.mark.parametrize("M", EPI_M)
def test_swiglu_epilogues_ragged_rows(ops, M):
    g = _gen(M + 1)
    D, Fh = 768, 2048
    x = _randn(g, M, D).to(bf16)
    w1 = (_randn(g, Fh, D) * D ** -0.5).to(bf16)
    w3 = (_randn(g, Fh, D) * D ** -0.5).to(bf16)
    w2 = (_randn(g, D, Fh) * Fh ** -0.5).to(bf16)
    dy = _randn(g, M, D).to(bf16)
    a, b = x.to(f64) @ w1.to(f64).t(), x.to(f64) @ w3.to(f64).t()
    ab, gate = ops.gemm_swiglu_fwd(x, interleave(w1, w3))
    abv = ab.view(M, Fh // 32, 2, 32)
    _check_bf16(abv[:, :, 0].reshape(M, Fh), a)
    _check_bf16(abv[:, :, 1].reshape(M, Fh), b)
    _check_bf16(gate, F.silu(a) * b)
    # backward on the stored (bf16) a, b
    a_s, b_s = abv[:, :, 0].reshape(M, Fh).to(f64), abv[:, :, 1].reshape(M, Fh).to(f64)
    dg = dy.to(f64) @ w2.to(f64)
    sg = torch.sigmoid(a_s)
    dab = ops.gemm_swiglu_bwd(dy, w2, ab).view(M, Fh // 32, 2, 32)
    _check_bf16(dab[:, :, 0].reshape(M, Fh), dg * b_s * (sg * (1 + a_s * (1 - sg))), 3e-2)
    _check_bf16(dab[:, :, 1].reshape(M, Fh), dg * a_s * sg, 3e-2)


@pytest.mark.parametrize("with_b1", [True, False])
@pytest.mark.parametrize("M", EPI_M)
def test_gelu_epilogues_ragged_rows(ops, M, with_b1):
    g = _gen(M + 2)
    D, N = 768, 3072
    x = _randn(g, M, D).to(bf16)
    w1 = (_randn(g, N, D) * 2 * D ** -0.5).to(bf16)
    b1 = torch.linspace(-3, 3, N, device="cuda") if with_b1 else None
    w2 = (_randn(g, D, N) * N ** -0.5).to(bf16)
    dy = _randn(g, M, D).to(bf16)
    uref = x.to(f64) @ w1.to(f64).t() + (b1.to(f64) if with_b1 else 0)
    u, h = ops.gemm_gelu_fwd(x, w1, b1)
    _check_bf16(u, uref)
    _check_bf16(h, F.gelu(uref))
    uu = u.to(f64).requires_grad_(True)
    F.gelu(uu).backward(dy.to(f64) @ w2.to(f64))
    _check_bf16(ops.gemm_gelu_bwd(dy, w2, u), uu.grad)


@pytest.mark.parametrize("V", [256, 64000])
@pytest.mark.parametrize("M", EPI_M)
def test_ce_ragged_rows(ops, M, V):
    """Fused head + cross-entropy partials and the dlogits chunk (tolerances of test_fused_head_cross_entropy)."""
    g = _gen(M + V)
    K = 768
    y = _randn(g, M, K).to(bf16)
    w = (_randn(g, V, K) * 0.05).to(bf16)
    tgt = torch.randint(0, V, (M,), device="cuda", generator=g)
    loss, lse = ops.ce_forward(y, w, tgt)
    v0, vc = (0, V) if V <= 1000 else (32000, 8000)
    gscale = torch.tensor([0.37], device="cuda")
    dl = torch.empty(M, vc, dtype=bf16, device="cuda")
    ops.ce_dlogits(y, w, tgt, lse, gscale, v0, vc, dl)
    ref_loss = 0.0
    for r0 in range(0, M, 4096):                                          # fp64 logits a row chunk at a time
        rs = slice(r0, min(M, r0 + 4096))
        logits = y[rs].to(f64) @ w.to(f64).t()
        ref_lse = torch.logsumexp(logits, -1)
        torch.testing.assert_close(lse[rs].to(f64), ref_lse, rtol=1e-5, atol=1e-4)
        ref_loss += F.cross_entropy(logits, tgt[rs], reduction="sum").item()
        p = torch.softmax(logits, -1)
        p[torch.arange(p.shape[0], device="cuda"), tgt[rs]] -= 1
        torch.testing.assert_close(dl[rs].to(f64), (p * 0.37)[:, v0:v0 + vc], rtol=2e-2, atol=1e-5)
    assert abs(loss.item() - ref_loss) <= 1e-5 * abs(ref_loss) + 1e-2
