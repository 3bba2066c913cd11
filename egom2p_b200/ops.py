"""Tensor-level wrappers over the C ABI: torch owns the memory and the stream, the library launches kernels.

Every function requires CUDA tensors and raises otherwise -- there is deliberately no CPU / eager fallback."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import torch

from . import _lib

bf16, f32 = torch.bfloat16, torch.float32


def _s() -> int:
    return torch.cuda.current_stream().cuda_stream


def _req_current(t: torch.Tensor):
    """Kernels are launched on the CURRENT device's current stream: a tensor living on another device would be addressed
    from the wrong context (ADVICE r1). Checked where tensors enter the library (`_req`)."""
    if t.device.index is not None and t.device.index != torch.cuda.current_device():
        raise RuntimeError(f"egom2p_b200: tensor on {t.device} but the current CUDA device is {torch.cuda.current_device()}; "
                           "wrap the call in torch.cuda.device(tensor.device)")


class KernelTimer:
    """Optional per-family CUDA-event timing (bench.py's roofline line). When active, wrappers bracket their launches
    with events on the current stream and record algorithmic work; `summary()` synchronises once at the end."""
    active: Optional["KernelTimer"] = None

    def __init__(self):
        self.records = []  # (family, work, unit, start_event, end_event)

    def __enter__(self):
        KernelTimer.active = self
        return self

    def __exit__(self, *exc):
        KernelTimer.active = None

    def summary(self):
        torch.cuda.synchronize()
        out: Dict[str, Dict[str, float]] = {}
        for fam, work, unit, e0, e1 in self.records:
            d = out.setdefault(fam, {"ms": 0.0, "work": 0.0, "launches": 0, "unit": unit})
            d["ms"] += e0.elapsed_time(e1)
            d["work"] += float(work)        # device scalars (mask-aware attention work) are read here, after the sync
            d["launches"] += 1
        return out


class _timed:
    __slots__ = ("fam", "work", "unit", "e0")

    def __init__(self, fam: str, work: float, unit: str):
        self.fam, self.work, self.unit = fam, work, unit

    def __enter__(self):
        if KernelTimer.active is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *exc):
        t = KernelTimer.active
        if t is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            t.records.append((self.fam, self.work, self.unit, self.e0, e1))


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, dtype, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"egom2p_b200: {name} must be a CUDA tensor (no CPU fallback exists)")
    if t.dtype != dtype:
        raise TypeError(f"egom2p_b200: {name} must be {dtype}, got {t.dtype}")
    _req_current(t)
    return t


def _req_dense(t: torch.Tensor, dtype, name: str, numel: Optional[int] = None):
    """_req plus the layout a kernel reads through a raw pointer: contiguous and, when given, `numel` elements."""
    _req(t, dtype, name)
    if not t.is_contiguous():
        raise ValueError(f"egom2p_b200: {name} must be contiguous (got strides {t.stride()} for shape {tuple(t.shape)})")
    if numel is not None and t.numel() != numel:
        raise ValueError(f"egom2p_b200: {name} must have {numel} elements, got shape {tuple(t.shape)}")
    return t


def _req_rows(t: torch.Tensor, dtype, name: str, cols: int):
    """A 2-D matrix of `cols` columns whose rows follow each other without a gap (row pitch == cols)."""
    _req(t, dtype, name)
    if t.dim() != 2 or t.shape[1] != cols or t.stride(1) != 1 or (t.shape[0] > 1 and t.stride(0) != cols):
        raise ValueError(f"egom2p_b200: {name} must be (rows, {cols}) with row pitch {cols}, got shape {tuple(t.shape)} "
                         f"and strides {t.stride()}")
    return t


# ----------------------------------------------------------------------------------------------- index plan
class Plan:
    """Outputs of egom2p_index_plan for one side (encoder or decoder)."""
    __slots__ = ("keep_idx", "keep_mod", "keep_pos", "pad", "mod_mask", "n_valid", "target_ids", "key_lo", "key_hi",
                 "B", "budget", "order", "row_batch", "rows", "slot_index", "slot_to_row")

    def __init__(self):
        self.row_batch = None   # packed plans: sample of every row (int32); None: rows are the (B, budget) slots
        self.rows = None        # packed plans: number of rows; None: B * budget


def index_plan(masks: Sequence[torch.Tensor], mod_ids: Sequence[int], budget: int, *, decoder: bool = False,
               attn_cnt: Optional[Sequence[torch.Tensor]] = None, ids: Optional[Sequence[torch.Tensor]] = None,
               causal: bool = False, sep: bool = True) -> Plan:
    lib = _lib.load()
    B = masks[0].shape[0]
    dev = masks[0].device
    d = _lib.PlanDesc()
    d.n_mods, d.batch, d.is_decoder, d.causal, d.sep = len(masks), B, int(decoder), int(causal), int(sep)
    keep = []
    total = 0
    for i, m in enumerate(masks):
        m = _req(m.reshape(B, -1), torch.bool, "mask").contiguous()
        keep.append(m)
        d.len[i], d.mod_id[i], d.mask[i] = m.shape[1], int(mod_ids[i]), m.data_ptr()
        total += m.shape[1]
        if decoder:
            a = _req(attn_cnt[i].reshape(B, -1), torch.int32, "decoder_attention_mask").contiguous()
            t = _req(ids[i].reshape(B, -1), torch.int64, "ids").contiguous()
            keep += [a, t]
            d.attn_cnt[i], d.ids[i] = a.data_ptr(), t.data_ptr()
    budget = min(int(budget), total)
    d.budget = budget
    pl = Plan()
    pl.B, pl.budget = B, budget
    pl.keep_idx = torch.empty(B, budget, dtype=torch.int32, device=dev)
    pl.keep_mod = torch.empty_like(pl.keep_idx)
    pl.keep_pos = torch.empty_like(pl.keep_idx)
    pl.pad = torch.empty(B, budget, dtype=torch.bool, device=dev)
    pl.mod_mask = torch.empty(B, budget, dtype=torch.int16, device=dev)
    pl.n_valid = torch.empty(B, dtype=torch.int32, device=dev)
    pl.target_ids = pl.key_lo = pl.key_hi = None
    if decoder:
        pl.target_ids = torch.empty(B, budget, dtype=torch.int64, device=dev)
        pl.key_lo = torch.empty(B, budget, dtype=torch.int32, device=dev)
        pl.key_hi = torch.empty_like(pl.key_lo)
    _lib.check(lib.egom2p_index_plan(C.byref(d), _p(pl.keep_idx), _p(pl.keep_mod), _p(pl.keep_pos), _p(pl.pad),
                                     _p(pl.mod_mask), _p(pl.n_valid), _p(pl.target_ids), _p(pl.key_lo), _p(pl.key_hi),
                                     _s()), "index_plan")
    return pl


def plan_rows(mod_mask: torch.Tensor, mod_ids: Sequence[int]):
    """Flat row indices of each modality id in `mod_mask` (any shape, int16): returns (rows (n_mods, total) int64 -- only the
    first counts[m] entries of row m are defined --, counts (n_mods,) int32), both on the device."""
    lib = _lib.load()
    _req(mod_mask, torch.int16, "mod_mask")
    flat = mod_mask.reshape(-1).contiguous()
    total, n = flat.numel(), len(mod_ids)
    rows = torch.empty(n, total, dtype=torch.int64, device=flat.device)
    counts = torch.empty(n, dtype=torch.int32, device=flat.device)
    ids = (C.c_int32 * n)(*[int(i) for i in mod_ids])
    _lib.check(lib.egom2p_plan_rows(_p(flat), total, ids, n, total, _p(rows), _p(counts), _s()), "plan_rows")
    return rows, counts


# ----------------------------------------------------------------------------------------------- embedding
def _embed_desc(B, dim, lens, vocabs, ids, tables, pos, mod):
    d = _lib.EmbedDesc()
    d.n_mods, d.dim = len(lens), dim
    for i in range(len(lens)):
        d.len[i], d.vocab[i] = lens[i], vocabs[i]
        if ids is not None:
            d.ids[i] = _req_dense(ids[i], torch.int64, "ids", B * lens[i]).data_ptr()
        if tables is not None:
            d.token_emb[i] = _req_dense(tables[i], f32, "token table", vocabs[i] * dim).data_ptr()
        d.pos_emb[i] = _req_dense(pos[i], f32, "pos_emb", lens[i] * dim).data_ptr()
        d.mod_emb[i] = _req_dense(mod[i], f32, "mod_emb", dim).data_ptr()
    return d


def embed_gather_fwd(plan: Plan, dim: int, lens, vocabs, ids, tables, pos, mod, mask_token=None, want_emb=True):
    lib = _lib.load()
    packed = plan.rows is not None
    rows = plan.rows if packed else plan.B * plan.budget
    dev = plan.keep_mod.device
    d = _embed_desc(plan.B, dim, lens, vocabs, ids, tables, pos, mod)
    if mask_token is not None:
        _req_dense(mask_token, f32, "mask_token", dim)
    x0 = torch.empty((rows, dim) if packed else (plan.B, plan.budget, dim), dtype=f32, device=dev)
    emb = torch.empty_like(x0) if want_emb else None
    with _timed("embed_gather", rows * dim * 4.0 * (2 + (1 if mask_token is None else 0) + (1 if want_emb else 0)), "byte"):
        _lib.check(lib.egom2p_embed_gather_fwd(C.byref(d), _p(mask_token), _p(plan.keep_mod), _p(plan.keep_pos), _p(plan.pad),
                                               _p(plan.row_batch), rows, plan.budget, _p(x0), _p(emb), _s()), "embed_gather_fwd")
    return x0, emb


def embed_gather_bwd(plan: Plan, dim: int, lens, vocabs, ids, pos, mod, dx0, demb, d_tables, d_mod, d_mask_token):
    lib = _lib.load()
    rows = plan.rows if plan.rows is not None else plan.B * plan.budget
    d = _embed_desc(plan.B, dim, lens, vocabs, ids, None, pos, mod)
    n = len(lens)
    _req_dense(dx0, f32, "dx0", rows * dim)
    if demb is not None:
        _req_dense(demb, f32, "demb", rows * dim)
    for i, t in enumerate(d_tables or []):
        if t is not None:
            _req_dense(t, f32, "d_tables", vocabs[i] * dim)
    for t in d_mod or []:
        if t is not None:
            _req_dense(t, f32, "d_mod", dim)
    if d_mask_token is not None:
        _req_dense(d_mask_token, f32, "d_mask_token", dim)
    arr_t = (C.c_void_p * _lib.MAX_MODS)(*[(_p(t) if t is not None else None) for t in (d_tables or [None] * n)])
    arr_m = (C.c_void_p * _lib.MAX_MODS)(*[(_p(t) if t is not None else None) for t in (d_mod or [None] * n)])
    _lib.check(lib.egom2p_embed_gather_bwd(C.byref(d), _p(dx0), _p(demb), _p(plan.keep_mod), _p(plan.keep_pos),
                                           _p(plan.pad), _p(plan.row_batch), rows, plan.budget, C.cast(arr_t, C.c_void_p),
                                           C.cast(arr_m, C.c_void_p), _p(d_mask_token), _s()), "embed_gather_bwd")


# ----------------------------------------------------------------------------------------------- layernorm
def layernorm_fwd(x: torch.Tensor, w: torch.Tensor, eps: float = 1e-6, out_bf16=True, out_f32=False, save_stats=True, bias=None):
    """bias: fp32 (D,) of a LayerNorm with a learnable bias (GELU / bias family), or None (no-bias kernel)."""
    lib = _lib.load()
    _req(x, f32, "x"); _req(w, f32, "weight")
    D = x.shape[-1]
    rows = x.numel() // D
    yb = torch.empty(x.shape, dtype=bf16, device=x.device) if out_bf16 else None
    yf = torch.empty_like(x) if out_f32 else None
    mean = torch.empty(rows, dtype=f32, device=x.device) if save_stats else None
    rstd = torch.empty(rows, dtype=f32, device=x.device) if save_stats else None
    with _timed("layernorm_fwd", rows * D * (4.0 + (2 if out_bf16 else 0) + (4 if out_f32 else 0)), "byte"):
        if bias is None:
            _lib.check(lib.egom2p_layernorm_fwd(_p(x), _p(w), rows, D, eps, _p(yb), _p(yf), _p(mean), _p(rstd), _s()), "layernorm_fwd")
        else:
            _req(bias, f32, "bias")
            _lib.check(lib.egom2p_layernorm_bias_fwd(_p(x), _p(w), _p(bias), rows, D, eps, _p(yb), _p(yf), _p(mean), _p(rstd), _s()),
                       "layernorm_bias_fwd")
    return yb, yf, mean, rstd


def layernorm_bwd(dy: torch.Tensor, x, w, mean, rstd, dx_in=None, d_weight=None, want_bf16=False, d_bias=None):
    """d_bias: fp32 (D,) accumulator of the bias gradient (sum of dy over rows) of a LayerNorm with a bias, or None."""
    lib = _lib.load()
    D = x.shape[-1]
    rows = x.numel() // D
    dx = torch.empty_like(x)
    dxb = torch.empty(x.shape, dtype=bf16, device=x.device) if want_bf16 else None
    dyb = dy if dy.dtype == bf16 else None
    dyf = dy if dy.dtype == f32 else None
    nbytes = rows * D * (4.0 + dy.element_size() + 4 + (4 if dx_in is not None else 0) + (2 if want_bf16 else 0))
    with _timed("layernorm_bwd", nbytes, "byte"):
        if d_bias is None:
            _lib.check(lib.egom2p_layernorm_bwd(_p(dyb), _p(dyf), _p(x), _p(w), _p(mean), _p(rstd), _p(dx_in), rows, D, _p(dx),
                                                _p(dxb), _p(d_weight), _s()), "layernorm_bwd")
        else:
            _req(d_bias, f32, "d_bias")
            _lib.check(lib.egom2p_layernorm_bias_bwd(_p(dyb), _p(dyf), _p(x), _p(w), _p(mean), _p(rstd), _p(dx_in), rows, D,
                                                     _p(dx), _p(dxb), _p(d_weight), _p(d_bias), _s()), "layernorm_bias_bwd")
    return dx, dxb


# ----------------------------------------------------------------------------------------------- GEMM
def gemm(A: torch.Tensor, B: torch.Tensor, M: int, N: int, K: int, *, a_mn=False, b_mn=False, bias=None, addend=None,
         out_bf16: Optional[torch.Tensor] = None, out_f32: Optional[torch.Tensor] = None):
    """C[M,N] = op(A) op(B)^T (+bias) (+addend). A/B are 2-D bf16 tensors with unit inner stride (views allowed)."""
    lib = _lib.load()
    _req(A, bf16, "A"); _req(B, bf16, "B")
    assert A.dim() == 2 and B.dim() == 2 and A.stride(1) == 1 and B.stride(1) == 1
    out = out_bf16 if out_bf16 is not None else out_f32
    assert out is not None and out.stride(-1) == 1
    ldc = out.stride(0)
    if out_bf16 is not None and out_f32 is not None:
        assert out_bf16.stride(0) == out_f32.stride(0)
    with _timed("gemm", 2.0 * M * N * K, "flop"):
        _lib.check(lib.egom2p_gemm_bf16(_p(A), _p(B), M, N, K, A.stride(0), B.stride(0), int(a_mn), int(b_mn), _p(bias),
                                        _p(addend), addend.stride(0) if addend is not None else 0, _p(out_bf16), _p(out_f32),
                                        ldc, _s()), "gemm_bf16")
    return out


def gemm_swiglu_fwd(x: torch.Tensor, w13: torch.Tensor):
    """ab = x @ w13^T (bf16, interleaved [a | b] groups of 32) and g = silu(a) * b, gate fused into the GEMM epilogue."""
    lib = _lib.load()
    R, K = x.shape
    N2 = w13.shape[0]
    ab = torch.empty(R, N2, dtype=bf16, device=x.device)
    g = torch.empty(R, N2 // 2, dtype=bf16, device=x.device)
    with _timed("gemm", 2.0 * R * N2 * K, "flop"):
        _lib.check(lib.egom2p_gemm_swiglu_fwd(_p(x), _p(w13), R, N2, K, x.stride(0), w13.stride(0), _p(ab), ab.stride(0), _p(g),
                                              g.stride(0), _s()), "gemm_swiglu_fwd")
    return ab, g


def gemm_swiglu_bwd(dy: torch.Tensor, w2: torch.Tensor, ab: torch.Tensor):
    """dab = swiglu'(ab) applied to dg = dy @ w2 inside the dgrad epilogue; w2 is (K, hidden) bf16."""
    lib = _lib.load()
    R, K = dy.shape
    hidden = w2.shape[1]
    dab = torch.empty(R, 2 * hidden, dtype=bf16, device=dy.device)
    with _timed("gemm", 2.0 * R * hidden * K, "flop"):
        _lib.check(lib.egom2p_gemm_swiglu_bwd(_p(dy), _p(w2), _p(ab), R, hidden, K, dy.stride(0), w2.stride(0), ab.stride(0),
                                              _p(dab), dab.stride(0), _s()), "gemm_swiglu_bwd")
    return dab


def gemm_gelu_fwd(x: torch.Tensor, w1: torch.Tensor, b1: Optional[torch.Tensor]):
    """u = x @ w1^T + b1 (bf16, saved for backward) and h = GELU(u) (bf16, exact erf form), activation fused into the epilogue."""
    lib = _lib.load()
    R, K = x.shape
    N = w1.shape[0]
    if b1 is not None:
        _req(b1, f32, "b1")
    u = torch.empty(R, N, dtype=bf16, device=x.device)
    h = torch.empty(R, N, dtype=bf16, device=x.device)
    with _timed("gemm", 2.0 * R * N * K, "flop"):
        _lib.check(lib.egom2p_gemm_gelu_fwd(_p(x), _p(w1), _p(b1), R, N, K, x.stride(0), w1.stride(0), _p(u), u.stride(0), _p(h),
                                            h.stride(0), _s()), "gemm_gelu_fwd")
    return u, h


def gemm_gelu_bwd(dy: torch.Tensor, w2: torch.Tensor, u: torch.Tensor):
    """du = GELU'(u) * (dy @ w2), the derivative applied inside the fc2 dgrad epilogue; w2 is (K, hidden) bf16."""
    lib = _lib.load()
    R, K = dy.shape
    hidden = w2.shape[1]
    du = torch.empty(R, hidden, dtype=bf16, device=dy.device)
    with _timed("gemm", 2.0 * R * hidden * K, "flop"):
        _lib.check(lib.egom2p_gemm_gelu_bwd(_p(dy), _p(w2), _p(u), R, hidden, K, dy.stride(0), w2.stride(0), u.stride(0), _p(du),
                                            du.stride(0), _s()), "gemm_gelu_bwd")
    return du


def linear_fwd(x: torch.Tensor, w: torch.Tensor, *, bias=None, addend=None, out_dtype=bf16):
    """y = x @ w^T, x (R,K) bf16, w (N,K) bf16."""
    R, K = x.shape
    N = w.shape[0]
    y = torch.empty(R, N, dtype=out_dtype, device=x.device)
    gemm(x, w, R, N, K, bias=bias, addend=addend, out_bf16=y if out_dtype == bf16 else None,
         out_f32=y if out_dtype == f32 else None)
    return y


def linear_dgrad(dy: torch.Tensor, w: torch.Tensor, *, addend=None, out_dtype=bf16):
    """dx = dy @ w, dy (R,N) bf16, w (N,K) bf16 (consumed MN-major, no transpose copy)."""
    R, N = dy.shape
    K = w.shape[1]
    dx = torch.empty(R, K, dtype=out_dtype, device=dy.device)
    gemm(dy, w, R, K, N, b_mn=True, addend=addend, out_bf16=dx if out_dtype == bf16 else None,
         out_f32=dx if out_dtype == f32 else None)
    return dx


def linear_wgrad(dy: torch.Tensor, x: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate=False):
    """dw = dy^T @ x, dy (R,N) bf16, x (R,K) bf16 -> (N,K) fp32 (both operands consumed MN-major)."""
    R, N = dy.shape
    K = x.shape[1]
    if out is None:
        out = torch.empty(N, K, dtype=f32, device=dy.device)
    gemm(dy, x, N, K, R, a_mn=True, b_mn=True, addend=out if accumulate else None, out_f32=out)
    return out


# ----------------------------------------------------------------------------------------------- head + CE
def ce_forward(y: torch.Tensor, w: torch.Tensor, target: torch.Tensor, keep_probs: bool = False):
    """Returns (loss_sum (1,) fp32, lse (R,) fp32) for logits = y @ w^T without materialising them.

    keep_probs (a head that needs a backward): the same pass also stores the softmax numerators, and the result gets a third
    item (probs (R, V) bf16, rscale (R,) fp32, tile_flag (ceil(R / 128),) uint8) with rscale[r] * probs[r, :] = softmax - onehot
    on the rows of unflagged 128-row tiles; a flagged tile's numerators are not exact in bf16, and `ce_dlogits(...,
    tile_flag=tile_flag)` recomputes them."""
    lib = _lib.load()
    _req(y, bf16, "y"); _req(w, bf16, "w")
    R, K = y.shape
    V = w.shape[0]
    _req_dense(target, torch.int64, "target", R)
    assert y.stride(1) == 1 and w.stride(1) == 1 and w.shape[1] == K
    nt = 2 * ((V + 255) // 256)  # two column halves per 256-wide vocabulary tile
    dev = y.device
    pm = torch.empty(nt, R, dtype=f32, device=dev)
    ps = torch.empty(nt, R, dtype=f32, device=dev)
    tl = torch.zeros(R, dtype=f32, device=dev)
    lse = torch.empty(R, dtype=f32, device=dev)
    loss = torch.zeros(1, dtype=f32, device=dev)
    if not keep_probs:
        with _timed("head_ce", 2.0 * R * V * K, "flop"):
            _lib.check(lib.egom2p_ce_partials(_p(y), _p(w), _p(target), R, V, K, y.stride(0), w.stride(0), _p(pm), _p(ps),
                                              _p(tl), _s()), "ce_partials")
        _lib.check(lib.egom2p_ce_finalize(_p(pm), _p(ps), _p(tl), R, nt, _p(lse), _p(loss), None, None, 0, None, 0, None, None,
                                          _s()), "ce_finalize")
        return loss, lse
    ref = torch.empty(R, dtype=f32, device=dev)
    wmax2 = torch.empty(1, dtype=f32, device=dev)
    probs = torch.empty(R, V, dtype=bf16, device=dev)
    rscale = torch.empty(R, dtype=f32, device=dev)
    tile_flag = torch.empty((R + 127) // 128, dtype=torch.uint8, device=dev)
    with _timed("head_ce", 2.0 * R * V * K, "flop"):
        _lib.check(lib.egom2p_ce_row_ref(_p(y), _p(w), R, V, K, y.stride(0), w.stride(0), _p(wmax2), _p(ref), _s()), "ce_row_ref")
        _lib.check(lib.egom2p_ce_probs(_p(y), _p(w), _p(target), _p(ref), R, V, K, y.stride(0), w.stride(0), _p(probs),
                                       probs.stride(0), _p(pm), _p(ps), _p(tl), _s()), "ce_probs")
    _lib.check(lib.egom2p_ce_finalize(_p(pm), _p(ps), _p(tl), R, nt, _p(lse), _p(loss), _p(ref), _p(target), V, _p(probs),
                                      probs.stride(0), _p(rscale), _p(tile_flag), _s()), "ce_finalize")
    return loss, lse, (probs, rscale, tile_flag)


def ce_dlogits(y, w, target, lse, gscale: Optional[torch.Tensor], v0: int, vc: int, out: torch.Tensor,
               tile_flag: Optional[torch.Tensor] = None):
    """out = (softmax - onehot) * gscale over the vocabulary columns [v0, v0 + vc) (gscale None: 1). With tile_flag (from
    ce_forward(keep_probs=True)) only the rows of flagged 128-row tiles are computed and written."""
    lib = _lib.load()
    R, K = y.shape
    if tile_flag is not None:
        _req_dense(tile_flag, torch.uint8, "tile_flag", (R + 127) // 128)
    with _timed("head_ce", 2.0 * R * vc * K, "flop"):
        _lib.check(lib.egom2p_ce_dlogits(_p(y), _p(w), _p(target), _p(lse), _p(gscale), _p(tile_flag), R, v0, vc, K, y.stride(0),
                                         w.stride(0), _p(out), out.stride(0), _s()), "ce_dlogits")
    return out


def ce_row_scale(y: torch.Tensor, rscale: torch.Tensor, gscale: torch.Tensor, want_ys: bool = True):
    """s = gscale * rscale (R,) fp32, and ys = bf16(s[:, None] * y) (R, K) when want_ys (else None)."""
    lib = _lib.load()
    _req(y, bf16, "y")
    R, K = y.shape
    _req_dense(rscale, f32, "rscale", R); _req_dense(gscale, f32, "gscale", 1)
    s = torch.empty(R, dtype=f32, device=y.device)
    ys = torch.empty(R, K, dtype=bf16, device=y.device) if want_ys else None
    _lib.check(lib.egom2p_ce_row_scale(_p(y), R, K, y.stride(0), _p(rscale), _p(gscale), _p(s), _p(ys), _s()), "ce_row_scale")
    return s, ys


# ----------------------------------------------------------------------------------------------- attention
def lse_stride(Mq: int) -> int:
    return int(_lib.load().egom2p_attn_lse_stride(Mq))


def attn_ranges(B, Mq, Nk, key_lo=None, key_hi=None, scale=None, device=None, empty_zero=False):
    """Range metadata of one (plan, attention kind), built once per forward and shared by all layers / heads.
    empty_zero: rows with an empty range get output 0 instead of uniform attention (inference only)."""
    lib = _lib.load()
    scale = (64 ** -0.5) if scale is None else scale
    device = device if device is not None else key_lo.device
    meta = torch.empty(lib.egom2p_attn_ranges_bytes(B, Mq), dtype=torch.uint8, device=device)
    _lib.check(lib.egom2p_attn_ranges(_p(key_lo), _p(key_hi), B, Mq, Nk, scale, int(empty_zero), _p(meta), _s()), "attn_ranges")
    return meta


def attn_fwd(q, k, v, B, H, Mq, Nk, key_lo=None, key_hi=None, scale=None, want_lse=True, meta=None, pairs=None):
    """q (B*Mq, >=H*64) / k, v (B*Nk, ...) bf16 2-D views with unit inner stride. Returns (o (B*Mq, H*64) bf16, lse).
    pairs: number of (query, key) pairs inside the ranges (host number or device scalar), for the timing breakdown only."""
    lib = _lib.load()
    if meta is None:
        meta = attn_ranges(B, Mq, Nk, key_lo, key_hi, scale, device=q.device)
    o = torch.empty(B * Mq, H * 64, dtype=bf16, device=q.device)
    lse = torch.empty(B, H, lse_stride(Mq), dtype=f32, device=q.device) if want_lse else None
    kmax = torch.empty(B * H, dtype=f32, device=q.device) if Nk > 0 else None   # scratch of the bound-path pre-pass
    with _timed("attn_fwd", 4.0 * H * 64 * (pairs if pairs is not None else B * Mq * Nk), "flop"):
        _lib.check(lib.egom2p_attn_fwd(_p(q), _p(k) if Nk > 0 else None, _p(v) if Nk > 0 else None, B, H, Mq, Nk, q.stride(0),
                                       k.stride(0) if Nk > 0 else 0, v.stride(0) if Nk > 0 else 0, _p(meta), _p(o),
                                       o.stride(0), _p(lse), _p(kmax), _s()), "attn_fwd")
    return o, lse


def attn_bwd(q, k, v, o, do, lse, B, H, Mq, Nk, dq, dk, dv, key_lo=None, key_hi=None, scale=None, meta=None, pairs=None):
    lib = _lib.load()
    scale = (64 ** -0.5) if scale is None else scale
    if meta is None:
        meta = attn_ranges(B, Mq, Nk, key_lo, key_hi, scale, device=q.device)
    assert do.stride(0) == o.stride(0)
    scratch = torch.empty(lib.egom2p_attn_bwd_scratch_bytes(B, H, Mq), dtype=torch.uint8, device=q.device)
    with _timed("attn_bwd", 10.0 * H * 64 * (pairs if pairs is not None else B * Mq * Nk), "flop"):
        _lib.check(lib.egom2p_attn_bwd(_p(q), _p(k), _p(v), _p(o), _p(do), _p(lse), B, H, Mq, Nk, q.stride(0), k.stride(0),
                                       v.stride(0), o.stride(0), _p(meta), scale, _p(scratch), _p(dq), _p(dk), _p(dv),
                                       dq.stride(0), dk.stride(0), dv.stride(0), _s()), "attn_bwd")


# ----------------------------------------------------------------------------------------------- elementwise
def cast_bf16(src: torch.Tensor, out: Optional[torch.Tensor] = None):
    lib = _lib.load()
    _req(src, f32, "src")
    src = src.contiguous()
    if out is None:
        out = torch.empty(src.shape, dtype=bf16, device=src.device)
    with _timed("cast", src.numel() * 6.0, "byte"):
        _lib.check(lib.egom2p_cast_f32_to_bf16(_p(src), _p(out), src.numel(), _s()), "cast_f32_to_bf16")
    return out


# Bumped by every backward of the model's autograd nodes (egom2p_b200/model.py): weights whose gradients were just produced are
# about to be rewritten by an optimizer, and torch's fused CUDA optimizers do not bump Tensor._version.
GRAD_GEN = [0]
_OPERAND_CACHE: Dict[int, tuple] = {}


def cached_bf16(weight: torch.Tensor) -> torch.Tensor:
    """bf16 GEMM operand of a standalone weight (the sampler-facing `nn.Linear` containers: vocabulary heads,
    decoder_proj_context), re-cast only when the master changed -- address, `_version`, or a backward since the last cast --
    instead of on every call (a 64k x 768 head is 295 MB of traffic per cast)."""
    w = weight.detach()
    key = id(weight)
    sig = (w.data_ptr(), weight._version, GRAD_GEN[0], tuple(w.shape))
    hit = _OPERAND_CACHE.get(key)
    if hit is not None and hit[0] == sig:
        return hit[1]
    wb = cast_bf16(w.contiguous())
    if len(_OPERAND_CACHE) > 64:
        _OPERAND_CACHE.clear()
    _OPERAND_CACHE[key] = (sig, wb)
    return wb


class CastPlan:
    """A fixed list of (fp32 master -> bf16 operand) casts run as ONE launch (egom2p_cast_f32_to_bf16_multi): the per-step
    refresh of the GEMM operands. items: (src (rows, cols) fp32 contiguous, dst bf16 2-D, group, slot)."""

    def __init__(self, items):
        import numpy as np
        dt = np.dtype([("src", "<u8"), ("dst", "<u8"), ("rows", "<i8"), ("first_chunk", "<i8"), ("cols", "<i4"), ("dst_ld", "<i4"),
                       ("group", "<i4"), ("slot", "<i4"), ("rows_per_chunk", "<i4"), ("pad", "<i4")])
        assert dt.itemsize == 56
        tab = np.zeros(len(items), dtype=dt)
        chunk = 0
        self.bytes = 0.0
        self.ptrs = []
        for i, (src, dst, group, slot) in enumerate(items):
            _req(src, f32, "src"); _req(dst, bf16, "dst")
            assert src.dim() == 2 and src.is_contiguous() and dst.dim() == 2 and dst.stride(1) == 1
            rows, cols = src.shape
            need_rows = rows if group == 0 else (rows + group - 1) // group * 2 * group
            assert dst.shape[0] >= need_rows and dst.shape[1] >= cols, "cast plan: destination too small"
            rpc = max(1, 8192 // cols)
            tab[i] = (src.data_ptr(), dst.data_ptr(), rows, chunk, cols, dst.stride(0), group, slot, rpc, 0)
            chunk += (rows + rpc - 1) // rpc
            self.bytes += rows * cols * 6.0
            self.ptrs.append((src.data_ptr(), dst.data_ptr()))
        self.n_items, self.n_chunks = len(items), chunk
        self.table = torch.from_numpy(tab.view(np.uint8).reshape(-1).copy()).to(items[0][0].device)

    def run(self):
        lib = _lib.load()
        with _timed("cast", self.bytes, "byte"):
            _lib.check(lib.egom2p_cast_f32_to_bf16_multi(_p(self.table), self.n_items, self.n_chunks, _s()), "cast_f32_to_bf16_multi")


def add_f32(a, b, want_f32=True, want_bf16=False):
    lib = _lib.load()
    out = torch.empty_like(a) if want_f32 else None
    outb = torch.empty(a.shape, dtype=bf16, device=a.device) if want_bf16 else None
    _lib.check(lib.egom2p_add_f32(_p(a), _p(b), a.numel(), _p(out), _p(outb), _s()), "add_f32")
    return out, outb


def colsum(x: torch.Tensor, out: torch.Tensor):
    lib = _lib.load()
    rows, cols = x.shape
    _lib.check(lib.egom2p_colsum_f32(_p(x), rows, cols, _p(out), _s()), "colsum_f32")
    return out


def colsum_bf16(x: torch.Tensor, out: Optional[torch.Tensor] = None):
    """Bias gradient out (+)= sum over rows of a bf16 (rows, cols) gradient (unit inner stride; views allowed)."""
    lib = _lib.load()
    _req(x, bf16, "x")
    assert x.dim() == 2 and x.stride(1) == 1
    rows, cols = x.shape
    if out is None:
        out = torch.zeros(cols, dtype=f32, device=x.device)
    if rows:
        with _timed("bias_grad", rows * cols * 2.0, "byte"):
            _lib.check(lib.egom2p_colsum_bf16(_p(x), rows, cols, x.stride(0), _p(out), _s()), "colsum_bf16")
    return out


def gather_rows_bf16(src: torch.Tensor, idx: torch.Tensor):
    """dst[i] = src[idx[i]]: src (rows, cols) bf16 with row pitch cols, idx int64 contiguous (every entry < rows)."""
    lib = _lib.load()
    _req_rows(src, bf16, "src", src.shape[-1])
    _req_dense(idx, torch.int64, "idx")
    n, cols = idx.numel(), src.shape[1]
    dst = torch.empty(n, cols, dtype=bf16, device=src.device)
    if n:
        _lib.check(lib.egom2p_gather_rows_bf16(_p(src), _p(idx), n, cols, _p(dst), _s()), "gather_rows_bf16")
    return dst


def scatter_rows_f32(src: torch.Tensor, idx: torch.Tensor, dst: torch.Tensor, row_scale: Optional[torch.Tensor] = None):
    """dst[idx[i]] = src[i] (times row_scale[i] when given, fp32 (n,)): src (n, cols) and dst (rows, cols) fp32 with row
    pitch cols, idx int64 contiguous (every entry < rows); rows of dst that idx does not name are left as they are."""
    lib = _lib.load()
    _req_rows(src, f32, "src", src.shape[-1])
    _req_rows(dst, f32, "dst", src.shape[1])
    _req_dense(idx, torch.int64, "idx", src.shape[0])
    if row_scale is not None:
        _req_dense(row_scale, f32, "row_scale", src.shape[0])
    n, cols = idx.numel(), src.shape[1]
    if n:
        _lib.check(lib.egom2p_scatter_rows_f32(_p(src), _p(idx), n, cols, _p(row_scale), _p(dst), _s()), "scatter_rows_f32")
    return dst


# ----------------------------------------------------------------------------------------------- generation
def sample_rows(logits: torch.Tensor, temperature: float, top_p: float = 0.0, top_k: int = 0, u: Optional[torch.Tensor] = None,
                want_prob: bool = True, want_kept: bool = False):
    """One token per row of fp32 logits (rows, V) with the reference's temperature / top-k / top-p semantics
    (generate.py:332-371). u: uniforms in [0, 1) per row (drawn with torch.rand on the current generator if None).
    Returns (token int64 (rows,), prob fp32 or None, n_kept int32 or None)."""
    lib = _lib.load()
    _req(logits, f32, "logits")
    assert logits.dim() == 2 and logits.stride(1) == 1
    rows, V = logits.shape
    if u is None:
        u = torch.rand(rows, device=logits.device, dtype=f32)
    _req(u, f32, "u")
    tok = torch.empty(rows, dtype=torch.int64, device=logits.device)
    prob = torch.empty(rows, dtype=f32, device=logits.device) if want_prob else None
    kept = torch.empty(rows, dtype=torch.int32, device=logits.device) if want_kept else None
    if rows:
        with _timed("sample", rows * V * 4.0, "byte"):
            _lib.check(lib.egom2p_sample_rows(_p(logits), logits.stride(0), rows, V, float(temperature), float(top_p), int(top_k),
                                              _p(u.contiguous()), _p(tok), _p(prob), _p(kept), _s()), "sample_rows")
    return tok, prob, kept


def cfg_combine_bf16(y_uncond: torch.Tensor, y_cond: torch.Tensor, scale: float) -> torch.Tensor:
    """bf16(y_u + (y_c - y_u) * scale) for fp32 tensors of equal shape (classifier-free guidance before the linear head)."""
    lib = _lib.load()
    _req(y_uncond, f32, "y_uncond"); _req(y_cond, f32, "y_cond")
    assert y_uncond.shape == y_cond.shape and y_uncond.is_contiguous() and y_cond.is_contiguous()
    out = torch.empty(y_uncond.shape, dtype=bf16, device=y_uncond.device)
    if out.numel():
        _lib.check(lib.egom2p_cfg_combine_bf16(_p(y_uncond), _p(y_cond), y_uncond.numel(), float(scale), _p(out), _s()), "cfg_combine_bf16")
    return out
