"""The vocabulary head's single-pass loss and backward (egom2p_b200.model._HeadLossFn over ops.ce_forward(keep_probs=True))
against fp64: loss, lse, dY (through decoder_norm) and dW.

The loss pass stores the softmax numerators P = 2^(l log2e - c_r) with c_r = ||y_r|| max_v ||w_v|| log2e; a row whose
largest logit is more than 60 (log2 units) below c_r is not exact in bf16, and its 128-row tile is recomputed by the backward.
Rows are forced there by a table row w* = 3 u of large norm: rows orthogonal to u have c_r - l_max log2e ~ 116, rows
along u have ~ 25. "valid" uses a random-init table (c_r ~ 25 everywhere), as the benchmark does."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

D = 768
GAIN = 1.7      # upstream gradient of the head's mean loss
L2E = 1.0 / math.log(2.0)


@pytest.fixture(scope="module")
def M():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from egom2p_b200 import model
    return model


def _bad_rows(R, mode):
    bad = torch.zeros(R, dtype=torch.bool)
    if mode == "invalid":
        bad[:] = True
    elif mode == "mixed":   # inside one 128-row tile, a whole tile, and the last (partial) tile
        bad[[r for r in (5, 77) if r < R]] = True
        if R > 12928:
            bad[12800:12928] = True
        bad[-1] = R > 128
    return bad


def _case(R, V, mode, seed=0):
    """y (S, D) fp32 (S > R: the head takes R of the rows, in a shuffled order), table w (V, D), rows idx, targets, bad rows."""
    g = torch.Generator(device="cuda").manual_seed(seed + R + V)
    S = R + 7
    y = torch.randn(S, D, generator=g, device="cuda", dtype=torch.float64)
    w = torch.randn(V, D, generator=g, device="cuda", dtype=torch.float64) * 0.02
    idx = torch.randperm(S, generator=g, device="cuda")[:R].contiguous()
    tgt = torch.randint(0, V, (R,), generator=g, device="cuda")
    bad = _bad_rows(R, mode)
    if mode != "valid":
        u = torch.randn(D, generator=g, device="cuda", dtype=torch.float64)
        u = u - u.mean()   # zero mean: the LayerNorm's centring leaves a row's component along u alone
        u = u / u.norm()
        w[V // 3] = 3 * u
        ym = y[idx]
        ym = ym - (ym @ u)[:, None] * u[None, :]                     # orthogonal to w*: the row is flagged
        good = ~bad.cuda()
        ym[good] += 37.0 * u                                          # along w*: exact, c_r - l_max log2e ~ 25
        y[idx] = ym
    return y.float(), w.float().bfloat16(), idx, tgt, bad


def _run(M, y, wb, idx, tgt, need_y=True, need_nw=True, need_w=True):
    yd = y.clone().requires_grad_(need_y)
    nw = torch.ones(D, device="cuda", requires_grad=need_nw)
    wt = wb.float().requires_grad_(need_w)
    losses = M._HeadLossFn.apply(yd, nw, None, [idx], [tgt], [wb], 1e-6, [0], True, wt)
    if need_y or need_nw or need_w:
        (losses[0] * GAIN).backward()
    torch.cuda.synchronize()
    return losses[0].detach(), yd.grad, nw.grad, wt.grad


def _reference(ops, y, wb, idx, tgt):
    """fp64 on the bf16 operands the kernels see (the LayerNorm kernel's bf16 output): mean loss, lse, dY, d(norm w), dW."""
    yn = ops.layernorm_fwd(y, torch.ones(D, device="cuda"), 1e-6)[0]
    ym, W = yn.index_select(0, idx).double(), wb.double()
    R = ym.shape[0]
    lse = torch.empty(R, dtype=torch.float64, device="cuda")
    dyn = torch.zeros(y.shape, dtype=torch.float64, device="cuda")
    dW = torch.zeros(W.shape, dtype=torch.float64, device="cuda")
    loss = 0.0
    for r0 in range(0, R, 2048):
        sl = slice(r0, min(R, r0 + 2048))
        logits = ym[sl] @ W.t()
        lse[sl] = torch.logsumexp(logits, -1)
        t = tgt[sl]
        loss += float((lse[sl] - logits.gather(1, t[:, None])[:, 0]).sum())
        G = torch.softmax(logits, -1)
        G[torch.arange(G.shape[0], device="cuda"), t] -= 1
        G *= GAIN / R
        dW += G.t() @ ym[sl]
        dyn[idx[sl]] = G @ W
        del logits, G
    y64 = y.double().requires_grad_(True)
    n64 = torch.ones(D, dtype=torch.float64, device="cuda", requires_grad=True)
    (F.layer_norm(y64, (D,), n64, None, 1e-6) * dyn).sum().backward()
    return loss / R, lse, y64.grad, n64.grad, dW, ym


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


CASES = [(R, V, mode) for R in (1, 129, 32288) for V in (256, 64000) for mode in ("valid", "invalid", "mixed")
         if not (R == 1 and mode == "mixed")]


@pytest.mark.parametrize("R,V,mode", CASES)
def test_head_single_pass_matches_fp64(M, R, V, mode):
    from egom2p_b200 import ops
    y, wb, idx, tgt, bad = _case(R, V, mode)
    loss_ref, lse_ref, dy_ref, dnw_ref, dw_ref, ym = _reference(ops, y, wb, idx, tgt)

    # the loss pass itself: lse, and which 128-row tiles fall back
    _, lse, (probs, rscale, tile_flag) = ops.ce_forward(ym.bfloat16(), wb, tgt, keep_probs=True)
    torch.testing.assert_close(lse.double(), lse_ref, rtol=1e-5, atol=1e-4)
    want = torch.zeros(tile_flag.numel(), dtype=torch.uint8)
    for r in torch.nonzero(bad)[:, 0].tolist():
        want[r // 128] = 1
    assert torch.equal(tile_flag.cpu(), want), (tile_flag.cpu().nonzero()[:, 0].tolist(), want.nonzero()[:, 0].tolist())
    del probs, rscale

    loss, dy, dnw, dw = _run(M, y, wb, idx, tgt)
    assert abs(float(loss) - loss_ref) <= 1e-5 * abs(loss_ref) + 1e-6, (float(loss), loss_ref)
    assert _rel(dw, dw_ref) < 5e-3, _rel(dw, dw_ref)
    assert _rel(dy, dy_ref) < 5e-3, _rel(dy, dy_ref)
    assert _rel(dnw, dnw_ref) < 5e-3, _rel(dnw, dnw_ref)
    rows = idx.cpu()
    for sel in (bad, ~bad):   # the fall-back rows and the single-pass rows each on their own
        if sel.any():
            r = rows[sel].cuda()
            assert _rel(dy[r], dy_ref[r]) < 5e-3, (sel.sum(), _rel(dy[r], dy_ref[r]))


@pytest.mark.parametrize("V", [256, 64000])
def test_head_frozen_and_no_dy(M, V):
    """A frozen head (no dW) and a head over a frozen trunk (want_dyn false: dW only) give the full backward's gradients."""
    from egom2p_b200 import ops
    y, wb, idx, tgt, bad = _case(1000, V, "mixed", seed=1)
    _, _, dy_ref, _, dw_ref, _ = _reference(ops, y, wb, idx, tgt)
    _, dy, dnw, dw = _run(M, y, wb, idx, tgt, need_w=False)
    assert dw is None and _rel(dy, dy_ref) < 5e-3
    _, dy, dnw, dw = _run(M, y, wb, idx, tgt, need_y=False, need_nw=False)
    assert dy is None and dnw is None and _rel(dw, dw_ref) < 5e-3


def test_head_no_grad_keeps_no_probs(M):
    from egom2p_b200 import ops
    y, wb, idx, tgt, _ = _case(129, 64000, "mixed", seed=2)
    loss_ref = _reference(ops, y, wb, idx, tgt)[0]
    with torch.no_grad():
        before = torch.cuda.memory_allocated()
        losses = M._HeadLossFn.apply(y, torch.ones(D, device="cuda"), None, [idx], [tgt], [wb], 1e-6, [0],
                                     torch.is_grad_enabled(), wb.float())
        held = torch.cuda.memory_allocated() - before
    assert held < 129 * 64000 * 2, held   # no (R, V) numerators kept
    assert abs(float(losses[0]) - loss_ref) <= 1e-5 * abs(loss_ref)


def test_head_step_under_graph_capture(M):
    """Forward + backward captured as one CUDA graph (the fall-back's tile gate is read on the device) replays to the
    eager step's loss and gradients."""
    y, wb, idx, tgt, _ = _case(1000, 64000, "mixed", seed=3)
    loss_e, dy_e, dnw_e, dw_e = _run(M, y, wb, idx, tgt)
    yd = y.clone().requires_grad_(True)
    nw = torch.ones(D, device="cuda", requires_grad=True)
    wt = wb.float().requires_grad_(True)

    def step():
        yd.grad = nw.grad = wt.grad = None
        loss = M._HeadLossFn.apply(yd, nw, None, [idx], [tgt], [wb], 1e-6, [0], True, wt)[0]
        (loss * GAIN).backward()
        return loss.detach()

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    yd.grad = nw.grad = wt.grad = None
    with torch.cuda.graph(graph):
        loss_g = step()
    graph.replay()
    torch.cuda.synchronize()
    assert abs(float(loss_g) - float(loss_e)) <= 1e-6 * abs(float(loss_e))
    for g, e in ((yd.grad, dy_e), (nw.grad, dnw_e), (wt.grad, dw_e)):
        assert _rel(g, e) < 1e-5, _rel(g, e)
