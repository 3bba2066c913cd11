"""GPU: training with frozen parameters. Every autograd node of the module (block, context, head and embedding functions)
computes only the gradients its inputs ask for (ctx.needs_input_grad): a frozen parameter gets neither a gradient nor the
work that would produce it. Checked on the tiny models of both families, dense and packed ragged batches, for each freeze
configuration below:

  * frozen parameters end the step with .grad None; every trainable parameter's gradient equals the one of the same step
    with nothing frozen (same weights, batch, decoder order) up to the run-to-run spread of the unfrozen step, and matches
    the CPU oracle with the tolerances of tests/test_model_gpu.py;
  * the skipped work is not launched: the weight-gradient GEMMs (ops.linear_wgrad), the bias column sums (ops.colsum_bf16),
    the head dW GEMMs and the context-side LayerNorm backwards are counted, and their number is the number of trainable
    consumers; the unfrozen step keeps the counts of the full backward.

Then a 3-step FusedAdamW trajectory under freeze_shared_params(), a CUDA-graph capture of a frozen model, unfreeze_all()
after a frozen step, and the LayerNorm-with-bias backward kernel with either reduction output left null."""
import ctypes as C
import math
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

import gelu_oracle as go  # noqa: E402
import synth  # noqa: E402
from test_gelu_family_gpu import _leaves as gelu_leaves  # noqa: E402
from test_gelu_family_gpu import build_gelu  # noqa: E402
from test_model_gpu import build_model, oracle_run, to_cuda  # noqa: E402

MODS4 = ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"]
N_ENC, N_DEC = 64, 48
BATCHES = {
    # every sample fills both budgets: slot layout, no pads
    "dense": dict(B=2, n_in={"tok_cam": [8, 8], "tok_depth": [24, 24], "tok_gaze": [8, 8], "tok_rgb": [24, 24]},
                  n_tgt={"tok_cam": [6, 6], "tok_depth": [18, 18], "tok_gaze": [6, 6], "tok_rgb": [18, 18]}),
    # ragged budgets: the rows are packed (valid tokens only)
    "ragged": dict(B=4, n_in={"tok_cam": [5, 1, 30, 2], "tok_depth": [30, 10, 0, 1], "tok_gaze": [4, 0, 30, 0], "tok_rgb": [25, 40, 4, 3]},
                   n_tgt={"tok_cam": [10, 30, 0, 1], "tok_depth": [20, 0, 40, 0], "tok_gaze": [3, 0, 0, 0], "tok_rgb": [15, 18, 70, 4]}),
}


def _freeze(mods, *params):
    for m in mods:
        for p in m.parameters():
            p.requires_grad = False
    for p in params:
        p.requires_grad = False


def _freeze_mlp_fc1(m):
    _freeze([], *[b.mlp.fc1.weight for b in (*m.encoder, *m.decoder)])


def _freeze_biases(m):
    _freeze([], *[p for n, p in m.named_parameters() if n.endswith(".bias")])


def _freeze_norm_weights(m):
    _freeze([], *[p for n, p in m.named_parameters() if "norm" in n and n.endswith(".weight")])


CONFIGS = {
    "shared": lambda m: m.freeze_shared_params(),
    "except_rgb_cam": lambda m: m.freeze_params_except_specific_embeddings("tok_rgb-tok_cam"),
    "encoder": lambda m: m.freeze_encoder(freeze_embeddings=True),
    # decoder-only training with decoder_proj_context frozen too: nothing upstream of the context trains, so no decoder
    # block computes the context gradient; context_norm still trains (its LayerNorm reduction alone runs)
    "encoder_and_context": lambda m: (m.freeze_encoder(freeze_embeddings=True), _freeze([m.decoder_proj_context])),
    "decoder": lambda m: m.freeze_decoder(freeze_embeddings=False),
    "one_block": lambda m: _freeze([m.decoder[0]]),
    # fc1 and fc3 share one interleaved wgrad GEMM (swiglu family): it still runs for fc3
    "mlp_fc1": _freeze_mlp_fc1,
}
GELU_CONFIGS = {
    "biases": _freeze_biases,               # Linear and LayerNorm biases frozen, weights trainable
    "norm_weights": _freeze_norm_weights,   # LayerNorm weights frozen, their biases trainable
}
CASES = [(fam, batch, cfg) for fam in ("swiglu", "gelu") for batch in BATCHES for cfg in CONFIGS if not (fam == "gelu" and cfg == "mlp_fc1")]
CASES += [("gelu", batch, cfg) for batch in BATCHES for cfg in GELU_CONFIGS]


def _family(fam):
    if fam == "swiglu":
        cfg = synth.make_cfg(192, 3, 2, 2, MODS4, video_vocab=512, video_thw=(5, 4, 4))
        return cfg, synth.make_state_dict(cfg, 5), build_model
    cfg = go.make_cfg(384, 6, 2, 2, MODS4, video_vocab=512, video_thw=(5, 4, 4))
    return cfg, go.make_state_dict(cfg, 5), build_gelu


def _model(fam, order):
    cfg, sd, build = _family(fam)
    model = build(cfg).cuda()
    model.load_state_dict(sd, strict=True)
    model.fixed_decoder_order = list(order)
    return model


def _batch(fam, name, seed=11):
    cfg = _family(fam)[0]
    return synth.make_batch(cfg, seed=seed, **BATCHES[name])


def _order():
    random.seed(3)
    return random.sample(MODS4, len(MODS4))


class _Counts:
    """Counts the launches of the gradient work that freezing can skip, by wrapping the ops the autograd nodes call:
    weight-gradient GEMMs, bias column sums, head dW GEMMs (an ops.gemm with an MN-major A outside linear_wgrad) and
    LayerNorm backwards over the context rows (decoder blocks' context_norm)."""

    def __init__(self):
        self.n = {"wgrad": 0, "colsum": 0, "head_dw": 0, "ctx_ln": 0}

    def __enter__(self):
        from egom2p_b200 import model as M
        from egom2p_b200 import ops
        self.ops, self.M = ops, M
        self.saved = {k: getattr(ops, k) for k in ("linear_wgrad", "colsum_bf16", "gemm", "layernorm_bwd")}
        inside, ctx_ptr = [False], [None]
        n, orig = self.n, self.saved

        def wgrad(*a, **k):
            n["wgrad"] += 1
            inside[0] = True
            try:
                return orig["linear_wgrad"](*a, **k)
            finally:
                inside[0] = False

        def colsum(*a, **k):
            n["colsum"] += 1
            return orig["colsum_bf16"](*a, **k)

        def gemm(*a, **k):
            n["head_dw"] += bool(k.get("a_mn")) and not inside[0]
            return orig["gemm"](*a, **k)

        def ln_bwd(dy, x, *a, **k):
            n["ctx_ln"] += ctx_ptr[0] is not None and x.data_ptr() == ctx_ptr[0]
            return orig["layernorm_bwd"](dy, x, *a, **k)

        apply = M._ContextFn.apply

        def ctx_apply(*a):
            out = apply(*a)
            ctx_ptr[0] = out.data_ptr()
            return out

        ops.linear_wgrad, ops.colsum_bf16, ops.gemm, ops.layernorm_bwd = wgrad, colsum, gemm, ln_bwd
        M._ContextFn.apply = staticmethod(ctx_apply)
        return self

    def __exit__(self, *exc):
        for k, v in self.saved.items():
            setattr(self.ops, k, v)
        del self.M._ContextFn.apply   # back to the inherited torch.autograd.Function.apply


def _step(model, md, counts=False):
    """One forward + backward; returns {name: grad or None} (and the launch counts)."""
    for p in model.parameters():
        p.grad = None
    if counts:
        with _Counts() as c:
            loss, _ = model(md, N_ENC, N_DEC)
            loss.backward()
    else:
        loss, _ = model(md, N_ENC, N_DEC)
        loss.backward()
    torch.cuda.synchronize()
    grads = {n: (None if p.grad is None else p.grad.detach().clone()) for n, p in model.named_parameters()}
    return (loss.item(), grads, c.n) if counts else (loss.item(), grads)


def _expected_counts(model, gelu):
    """Launches of the skippable gradient work that the trainable parameters ask for."""
    rg = lambda p: bool(p.requires_grad)
    n = {"wgrad": 0, "colsum": 0, "head_dw": 0, "ctx_ln": 0}

    def lin(*ls):
        for layer in ls:
            n["wgrad"] += rg(layer.weight)
            n["colsum"] += layer.bias is not None and rg(layer.bias)

    def mlp(m):
        if gelu:
            lin(m.fc1, m.fc2)
        else:
            n["wgrad"] += (rg(m.fc1.weight) or rg(m.fc3.weight)) + rg(m.fc2.weight)

    for b in model.encoder:
        lin(b.attn.qkv, b.attn.proj)
        mlp(b.mlp)
    upstream = [*model.encoder_embeddings.parameters(), *model.encoder.parameters(), *model.encoder_norm.parameters(),
                *model.decoder_proj_context.parameters()]
    ctx_grad = any(rg(p) for p in upstream)
    n["wgrad"] += ctx_grad and rg(model.decoder_proj_context.weight)
    for b in model.decoder:
        lin(b.self_attn.qkv, b.self_attn.proj, b.cross_attn.q, b.cross_attn.kv, b.cross_attn.proj)
        mlp(b.mlp)
        n["ctx_ln"] += ctx_grad or any(rg(p) for p in b.context_norm.parameters())
    for e in model.decoder_embeddings.values():   # every modality of the test batches has targets
        n["head_dw"] += rg(e.to_logits.weight) * math.ceil(e.to_logits.weight.shape[0] / 8192)
    return n


def _full_counts(model, gelu):
    """Counts of the backward with every parameter trainable: per encoder block qkv, proj and the two MLP GEMMs, per decoder
    block three more (q, kv, cross proj); plus decoder_proj_context; one bias sum per Linear of the GELU family."""
    E, D = len(model.encoder), len(model.decoder)
    return {"wgrad": 4 * E + 7 * D + 1, "colsum": (4 * E + 7 * D) if gelu else 0, "head_dw": len(model.decoder_embeddings),
            "ctx_ln": D}


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


_REF = {}


def _reference(fam, batch):
    """The unfrozen step, twice (its run-to-run spread), and the oracle's gradients, for one family and batch."""
    key = (fam, batch)
    if key not in _REF:
        order = _order()
        md = _batch(fam, batch)
        model = _model(fam, order)
        mdc = to_cuda(md)
        loss, g1, counts = _step(model, mdc, counts=True)
        _, g2 = _step(model, mdc)
        assert counts == _full_counts(model, fam == "gelu"), counts
        # dQ of the attention backward and the embedding / LayerNorm reductions add fp32 partials with atomics, in an order
        # that varies from run to run: the spread of two identical unfrozen steps is the scale of the noise
        spread = max(_rel(g1[n], g2[n]) for n in g1 if g1[n] is not None)
        cfg, sd, _ = _family(fam)
        if fam == "swiglu":
            _, leaf = oracle_run(sd, cfg, md, N_ENC, N_DEC, order)
        else:
            leaf = gelu_leaves(sd, cfg)
            go.forward(leaf, cfg, md, N_ENC, N_DEC, dec_order=order, keep=True)["loss"].backward()
        _REF[key] = (loss, g1, spread, {n: t.grad for n, t in leaf.items()})
    return _REF[key]


@pytest.mark.parametrize("fam,batch,config", CASES)
def test_frozen_step(fam, batch, config):
    loss_ref, g_ref, spread, g_orc = _reference(fam, batch)
    model = _model(fam, _order())
    {**CONFIGS, **GELU_CONFIGS}[config](model)
    frozen = {n for n, p in model.named_parameters() if not p.requires_grad}
    assert frozen and len(frozen) < len(g_ref)
    loss, grads, counts = _step(model, to_cuda(_batch(fam, batch)), counts=True)
    assert abs(loss - loss_ref) <= 1e-6 * abs(loss_ref), (loss, loss_ref)
    assert counts == _expected_counts(model, fam == "gelu"), (counts, _expected_counts(model, fam == "gelu"))
    # the bound: ten times the largest relative spread of two unfrozen steps, at least 1e-4 (the same kernels add the same
    # terms; only the order of the atomic fp32 sums differs). The oracle tolerances below are 300 times looser.
    bound = max(10 * spread, 1e-4)
    bad = []
    for name, g in grads.items():
        if name in frozen:
            assert g is None, f"frozen {name} got a gradient"
            continue
        assert g is not None and torch.isfinite(g).all(), name
        err = _rel(g, g_ref[name])
        if err > bound:
            bad.append((name, err, bound))
        if g_orc[name] is not None:
            tol = 5e-2 if ("cross_attn.q." in name or "query_norm" in name) else 3e-2
            err_o = _rel(g.cpu(), g_orc[name])
            if err_o > tol:
                bad.append((name, "oracle", err_o, tol))
    assert not bad, bad


def test_adamw_trajectory_under_freeze_shared_params():
    """Three FusedAdamW steps (clip 1.0) of a model under freeze_shared_params() against three steps of an unfrozen model
    whose gradients of the same parameters are dropped before each step: the frozen weights stay bitwise unchanged, the
    trainable ones follow the same trajectory."""
    from egom2p_b200.optim import FusedAdamW
    order = _order()
    batches = [to_cuda(_batch("swiglu", "ragged", seed=50 + i)) for i in range(3)]
    frozen_model, full_model = _model("swiglu", order), _model("swiglu", order)
    frozen_model.freeze_shared_params()
    names = {n for n, p in frozen_model.named_parameters() if not p.requires_grad}
    init = {n: p.detach().clone() for n, p in frozen_model.named_parameters()}
    lr = 3e-3
    mk = lambda m: FusedAdamW([{"params": list(m.parameters()), "weight_decay": 0.05}], lr=lr, betas=(0.9, 0.95))
    opts = [mk(frozen_model), mk(full_model)]
    for md in batches:
        losses = []
        for model, opt in zip((frozen_model, full_model), opts):
            loss, _ = model(md, N_ENC, N_DEC)
            loss.backward()
            if model is full_model:
                for n, p in model.named_parameters():
                    if n in names:
                        p.grad = None
            opt.clip_grad_norm_(1.0)
            opt.step()
            opt.zero_grad(set_to_none=True)
            losses.append(loss.item())
        assert abs(losses[0] - losses[1]) <= 2e-4 * abs(losses[1]), losses
    torch.cuda.synchronize()
    lr_sum = 3 * lr
    full = dict(full_model.named_parameters())
    for n, p in frozen_model.named_parameters():
        if n in names:
            assert torch.equal(p.detach(), init[n]), n
            continue
        assert not torch.equal(p.detach(), init[n]), n
        # as in tests/test_train_steps_gpu.py: Adam moves every element by about lr whatever its gradient's size, so an
        # element whose gradient is near zero may step either way in two runs whose fp32 atomics differ in the last bits
        d = (p.detach() - full[n].detach()).abs()
        assert d.max().item() <= 2.2 * lr_sum and d.mean().item() <= 0.05 * lr_sum, (n, d.max().item(), d.mean().item())


def test_graphed_step_on_frozen_model():
    from egom2p_b200.graphed import GraphedTrainStep
    from egom2p_b200.optim import FusedAdamW
    n_in = {"tok_cam": [5, 30], "tok_depth": [30, 10], "tok_gaze": [4, 3], "tok_rgb": [25, 21]}
    n_tg = {"tok_cam": [10, 3], "tok_depth": [20, 7], "tok_gaze": [3, 7], "tok_rgb": [15, 18]}
    cfg, sd, _ = _family("swiglu")
    batches = [to_cuda(synth.make_batch(cfg, B=2, seed=30 + i, n_in=n_in, n_tgt=n_tg)) for i in range(2)]
    eager, graphed = _model("swiglu", _order()), _model("swiglu", _order())
    for m in (eager, graphed):
        m.freeze_shared_params()
    mk = lambda m: FusedAdamW([{"params": [p for p in m.parameters() if p.requires_grad], "weight_decay": 0.05}], lr=1e-3,
                              betas=(0.9, 0.95))
    o_e, o_g = mk(eager), mk(graphed)
    runner = GraphedTrainStep(graphed, o_g, batches[1], N_ENC, N_DEC, clip_grad=1.0)
    eager.fixed_decoder_order = list(graphed.fixed_decoder_order)
    frozen = {n: p.detach().clone() for n, p in graphed.named_parameters() if not p.requires_grad}
    for md in batches:
        loss_e, _ = eager(md, N_ENC, N_DEC)
        loss_e.backward()
        o_e.clip_grad_norm_(1.0)
        o_e.step()
        o_e.zero_grad(set_to_none=True)
        loss_g = runner(md)
        torch.cuda.synchronize()
        assert abs(loss_e.item() - loss_g.item()) <= 2e-4 * abs(loss_e.item()), (loss_e.item(), loss_g.item())
    for n, p in graphed.named_parameters():
        if n in frozen:
            assert torch.equal(p.detach(), frozen[n]) and p.grad is None, n


@pytest.mark.parametrize("fam", ["swiglu", "gelu"])
def test_unfreeze_all_restores_full_gradients(fam):
    _, g_ref, spread, _ = _reference(fam, "dense")
    model = _model(fam, _order())
    md = to_cuda(_batch(fam, "dense"))
    model.freeze_shared_params()
    _step(model, md)
    model.unfreeze_all()
    _, grads, counts = _step(model, md, counts=True)
    assert counts == _full_counts(model, fam == "gelu"), counts
    bound = max(10 * spread, 1e-4)
    for name, g in grads.items():
        assert g is not None, name
        assert _rel(g, g_ref[name]) <= bound, (name, _rel(g, g_ref[name]), bound)


@pytest.mark.parametrize("null", ["d_weight", "d_bias", "both"])
def test_layernorm_bias_bwd_with_null_reduction(null):
    """The LayerNorm-with-bias backward kernel leaves a null d_weight or d_bias (a frozen parameter) unreduced and
    computes the other outputs exactly as with both present."""
    from egom2p_b200 import _lib, ops
    R, dim = 1000, 384
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(R, dim, device="cuda", generator=g) * 2 + 0.5
    w = 1 + 0.1 * torch.randn(dim, device="cuda", generator=g)
    b = 0.1 * torch.randn(dim, device="cuda", generator=g)
    dy = torch.randn(R, dim, device="cuda", generator=g)
    _, _, mean, rstd = ops.layernorm_fwd(x, w, 1e-6, bias=b)
    dw_ref, db_ref = torch.zeros(dim, device="cuda"), torch.zeros(dim, device="cuda")
    dx_ref, _ = ops.layernorm_bwd(dy, x, w, mean, rstd, d_weight=dw_ref, d_bias=db_ref)
    dw = None if null in ("d_weight", "both") else torch.zeros(dim, device="cuda")
    db = None if null in ("d_bias", "both") else torch.zeros(dim, device="cuda")
    dx = torch.empty_like(x)
    p = lambda t: None if t is None else t.data_ptr()
    lib = _lib.load()
    _lib.check(lib.egom2p_layernorm_bias_bwd(None, dy.data_ptr(), x.data_ptr(), w.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                             None, R, dim, dx.data_ptr(), None, p(dw), p(db),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)), "layernorm_bias_bwd")
    torch.cuda.synchronize()
    assert torch.equal(dx, dx_ref)
    if dw is not None:
        torch.testing.assert_close(dw, dw_ref, rtol=1e-5, atol=1e-4)
    if db is not None:
        torch.testing.assert_close(db, db_ref, rtol=1e-5, atol=1e-4)
