"""GPU: egom2p_b200.optim.FusedAdamW (egom2p_sumsq_multi + egom2p_adamw_multi_steps) against torch.optim.AdamW(foreach=False) and
torch.nn.utils.clip_grad_norm_ run in fp64 on the device, on fp64 copies of the SAME fp32 gradients the kernels read. Both sides
get identical inputs, so what is left is the kernels' fp32 arithmetic, and the tolerances follow from it:

  * gradient norm: fp32 partial sums of at most 8192 squares, added in fp64 -> rtol 1e-5;
  * exp_avg_sq: a sum of positive terms, relative error a few fp32 ulps per step plus twice the clip coefficient's
    (~1e-6) -> rtol 1e-5; exp_avg can cancel, so it also gets an absolute 1e-5 of the largest gradient the tensor saw;
  * parameters: a step rounds twice on |p| (the decay product, whose fp32 factor 1 - lr * wd carries at most one ulp of |p|,
    and the update), <= 2 ulp(|p|), and the update lr * m_hat / (sqrt(v_hat) + eps) is right to ~1e-6 relative
    (scale-free in the gradient, so the clip coefficient's error cancels) -> per element, after n steps with learning
    rates summing to L: n * 2 * ulp(|p| + L) + 1e-5 * L.

Every way of getting the step count, the bias correction or the clip coefficient wrong moves a parameter by a sizeable
fraction of lr, orders of magnitude above these bounds. Each comparison prints its largest error as a fraction of the
bound (pytest -s)."""
import io
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

import synth  # noqa: E402

BETAS, EPS = (0.9, 0.95), 1e-8
EDGE_SIZES = [1, 3, 4, 8191, 8192, 8193, 16385]


@pytest.fixture(scope="module")
def optim():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from egom2p_b200 import optim as _optim
    return _optim


class Pair:
    """A FusedAdamW over fp32 parameters and a torch.optim.AdamW(foreach=False) over fp64 copies, with the same groups."""

    def __init__(self, optim, groups, lr=1e-3):
        self.p32 = [p for ps, _ in groups for p in ps]
        self.p64 = [p.detach().double().clone() for p in self.p32]
        self.fused = optim.FusedAdamW([{"params": ps, "weight_decay": wd} for ps, wd in groups], lr=lr, betas=BETAS, eps=EPS)
        it = iter(self.p64)
        self.ref = torch.optim.AdamW([{"params": [next(it) for _ in ps], "weight_decay": wd} for ps, wd in groups], lr=lr,
                                     betas=BETAS, eps=EPS, foreach=False)
        self.gmax = [0.0] * len(self.p32)
        self.n_steps, self.lr_sum = 0, 0.0

    def step(self, grads, lrs, wds=None, max_norm=None):
        """One step of both with `grads` (fp32 device tensors, None = no gradient); returns (fused norm, fp64 norm)."""
        for opt in (self.fused, self.ref):
            for i, g in enumerate(opt.param_groups):
                g["lr"] = lrs[i]
                if wds is not None:
                    g["weight_decay"] = wds[i]
        for i, (a, b, g) in enumerate(zip(self.p32, self.p64, grads)):
            a.grad = g
            b.grad = None if g is None else g.double()
            if g is not None:
                self.gmax[i] = max(self.gmax[i], g.abs().nan_to_num(posinf=0.0).max().item())
        n32 = n64 = None
        if max_norm is not None:
            n32 = self.fused.clip_grad_norm_(max_norm)
            n64 = torch.nn.utils.clip_grad_norm_([p for p in self.p64 if p.grad is not None], max_norm, foreach=False)
        self.fused.step()
        self.ref.step()
        self.n_steps += 1
        self.lr_sum += max(lrs)
        return n32, n64

    def check(self, what, p32=None, state32=None):
        """Parameters, moments and per-tensor step counts of the fused side (or of `p32` / `state32`, a continuation of it)
        against the fp64 side; returns the largest parameter error as a fraction of its bound."""
        p32 = self.p32 if p32 is None else p32
        state32 = self.fused.state if state32 is None else state32
        worst = 0.0
        for i, (a, b) in enumerate(zip(p32, self.p64)):
            sa, sb = state32[a], self.ref.state[b]
            assert bool(sa) == bool(sb), (what, i)
            if not sb:
                assert torch.equal(a.detach().double(), b.detach()), (what, i)
                continue
            worst = max(worst, _param_err(a, b, self.n_steps, self.lr_sum, f"{what}: tensor {i} {tuple(a.shape)}"))
            torch.testing.assert_close(sa["exp_avg"].double(), sb["exp_avg"], rtol=1e-5, atol=1e-5 * self.gmax[i], equal_nan=True,
                                       msg=lambda m: f"{what}: exp_avg of tensor {i}: {m}")
            torch.testing.assert_close(sa["exp_avg_sq"].double(), sb["exp_avg_sq"], rtol=1e-5, atol=0, equal_nan=True,
                                       msg=lambda m: f"{what}: exp_avg_sq of tensor {i}: {m}")
            assert int(sa["step"]) == int(sb["step"]), (what, i, int(sa["step"]), int(sb["step"]))
        print(f"{what}: largest parameter error {worst:.3f} of the bound")
        return worst


def _param_err(a, b, n_steps, lr_sum, what):
    a, b = a.detach(), b.detach()
    nan = torch.isnan(b)
    assert torch.equal(torch.isnan(a), nan), f"{what}: NaN pattern differs"
    top = (b.abs() + lr_sum).float().nan_to_num(nan=1.0)
    ulp = (torch.nextafter(top, torch.full_like(top, float("inf"))) - top).double()
    bound = n_steps * 2 * ulp + 1e-5 * lr_sum
    r = ((a.double() - b).abs() / bound).masked_fill(nan, 0.0).max().item()
    assert r <= 1.0, f"{what}: parameter error {r:.3g} x the bound"
    return r


def _randn(shape, gen, scale=1.0):
    return torch.randn(shape, generator=gen, device="cuda") * scale


def _norm64(grads):
    return torch.stack([g.double().norm() for g in grads if g is not None]).norm().item()


# ------------------------------------------------------------------------------------------ 1. the full ego-b table
def test_full_size_table(optim, golden_dir):
    """All 245 ego-b tensors in bench.py's two weight-decay groups, 3 steps with a per-step lr / weight decay, per-tensor
    gradient scales, all-zero embedding rows, and the clip active on steps 0 and 2 only. The table has > 1024 chunks, so the
    single-block finalize of the norm strides."""
    man = json.load(open(os.path.join(golden_dir, "egob_state_dict_manifest.json")))
    shapes = {n: man["state_dict"][n] for n in man["named_parameters"]}
    assert len(shapes) == 245
    gen = torch.Generator(device="cuda").manual_seed(0)
    params = {}
    for n, s in shapes.items():
        params[n] = (1.0 + _randn(s, gen, 0.1)) if "norm" in n and n.endswith("weight") else _randn(s, gen, 0.02)
    decay = [p for n, p in params.items() if not ("norm" in n or n.endswith(".bias"))]
    no_decay = [p for n, p in params.items() if "norm" in n or n.endswith(".bias")]
    pair = Pair(optim, [(decay, 0.05), (no_decay, 0.0)])
    names = [n for n, p in params.items() if not ("norm" in n or n.endswith(".bias"))] + \
            [n for n, p in params.items() if "norm" in n or n.endswith(".bias")]
    scales = 10.0 ** (torch.arange(len(names), dtype=torch.float64) % 7 - 4.0)       # 1e-4 .. 1e2, per tensor
    for t, active in enumerate([True, False, True]):
        grads = []
        for n, p, sc in zip(names, pair.p32, scales.tolist()):
            g = _randn(p.shape, gen, sc)
            if "token_emb" in n:
                g[3::5] = 0.0                   # vocabulary rows no token uses: zero moments, an update of 0 / (0 + eps)
            grads.append(g)
        norm = _norm64(grads)
        max_norm = 0.5 * norm if active else 2.0 * norm
        n32, n64 = pair.step(grads, lrs=[1e-3 * (1 + t), 1e-3 * (1 + t)], wds=[0.05 * (1 - 0.3 * t), 0.0], max_norm=max_norm)
        torch.testing.assert_close(n32.double().cpu(), n64.cpu(), rtol=1e-5, atol=0)
        del grads
    assert pair.fused._n_chunks > 1024, pair.fused._n_chunks
    pair.check("full-size table")


# ------------------------------------------------------------------------------------------ 2. chunk and alignment edges
@pytest.mark.parametrize("layout", ["separate", "grad_views", "param_views"])
def test_chunk_and_alignment_edges(optim, layout):
    """Tensors of 1, 3, 4, 8191, 8192, 8193 and 16385 elements, separately allocated, or with the gradients (or the params)
    as contiguous views at element offsets 1..3 of one flat buffer, as DDP's gradient_as_bucket_view lays gradients out.
    The views reach the scalar paths of both kernels, which every ego-b tensor (a multiple of 4, 16-byte aligned) skips."""
    gen = torch.Generator(device="cuda").manual_seed(1)

    def views(sizes, fill):
        flat = torch.empty(sum(sizes) + 7 * len(sizes), device="cuda")
        out, pos = [], 0
        for i, n in enumerate(sizes):
            pos = (pos + 3) // 4 * 4 + 1 + i % 3
            v = flat[pos:pos + n]
            v.copy_(fill(n))
            out.append(v)
            pos += n
        assert all(v.data_ptr() % 16 for v in out)
        return out

    sizes = EDGE_SIZES + EDGE_SIZES[::-1]
    init = lambda n: _randn(n, gen, 0.02)
    ps = views(sizes, init) if layout == "param_views" else [init(n) for n in sizes]
    half = len(ps) // 2
    pair = Pair(optim, [(ps[:half], 0.05), (ps[half:], 0.0)])
    for t, active in enumerate([True, False, True]):
        mk = lambda n: _randn(n, gen, 3.0 if active else 1e-3)
        grads = views(sizes, mk) if layout == "grad_views" else [mk(n) for n in sizes]
        max_norm = 0.5 * _norm64(grads) if active else 1.0
        n32, n64 = pair.step(grads, lrs=[1e-3 * (1 + t), 2e-3], max_norm=max_norm)
        torch.testing.assert_close(n32.double().cpu(), n64.cpu(), rtol=1e-5, atol=0)
    pair.check(f"edges ({layout})")


# ------------------------------------------------------------------------------------------ 3. late and skipped gradients
def test_late_and_skipped_gradients(optim):
    """Group A has gradients from step 1; group B has none for 5 steps (frozen) and then gets them (unfrozen); one tensor of
    group A sits out step 4. As in torch, a tensor without a gradient takes no step: its first update after the pause
    uses its own step count, so group B's first bias correction is t = 1, not 6."""
    gen = torch.Generator(device="cuda").manual_seed(2)
    a = [_randn(n, gen, 0.02) for n in (8192, 300, 16385)]
    b = [_randn(n, gen, 0.02) for n in (4096, 8193)]
    pair = Pair(optim, [(a, 0.05), (b, 0.05)])
    for t in range(10):
        grads = [_randn(p.shape, gen) for p in pair.p32]
        if t < 5:
            grads[3] = grads[4] = None
        if t == 4:
            grads[1] = None
        pair.step(grads, lrs=[1e-3, 1e-3], max_norm=1.0 if t % 2 else None)
    pair.check("late / skipped gradients")
    assert [int(pair.fused.state[p]["step"]) for p in pair.p32] == [10, 9, 10, 5, 5]


def test_frozen_blocks_get_no_gradient():
    """The scenario above arises in training: after freeze_shared_params() a backward through the block autograd functions
    leaves every encoder / decoder block parameter's .grad None, while the embeddings get gradients."""
    from test_model_gpu import build_model, to_cuda
    cfg = synth.make_cfg(192, 3, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=512, video_thw=(5, 4, 4))
    md = to_cuda(synth.make_batch(cfg, B=2, seed=41, n_in={"tok_cam": [5, 30], "tok_depth": [30, 10], "tok_gaze": [4, 3], "tok_rgb": [25, 21]},
                                  n_tgt={"tok_cam": [10, 3], "tok_depth": [20, 7], "tok_gaze": [3, 7], "tok_rgb": [15, 18]}))
    model = build_model(cfg).cuda()
    model.load_state_dict(synth.make_state_dict(cfg, 4), strict=True)
    model.freeze_shared_params()
    loss, _ = model(md, 64, 48)
    loss.backward()
    shared = [(n, p) for n, p in model.named_parameters() if n.split(".")[0] in ("encoder", "decoder", "encoder_norm", "decoder_norm")]
    assert shared and all(p.grad is None for _, p in shared), [n for n, p in shared if p.grad is not None]
    assert any(p.grad is not None for n, p in model.named_parameters() if "embeddings" in n)


# ------------------------------------------------------------------------------------------ 4. resume
def _table(gen, sizes=(8192, 5, 16385, 768, 3000)):
    return [_randn(n, gen, 0.02) for n in sizes]


def _roundtrip(sd):
    buf = io.BytesIO()
    torch.save(sd, buf)
    buf.seek(0)
    return torch.load(buf, map_location="cpu")


def test_resume_is_bitwise(optim):
    """k steps, state_dict -> torch.save -> torch.load -> a fresh FusedAdamW -> load_state_dict -> k more steps gives bitwise
    the parameters and moments of 2k uninterrupted steps: both kernels are elementwise or fixed-order sums. The saved form is
    torch's: an independent float32 CPU step per tensor."""
    k = 3
    gen = torch.Generator(device="cuda").manual_seed(3)
    p0 = _table(gen)
    grads = [[_randn(p.shape, gen) for p in p0] for _ in range(2 * k)]
    groups = lambda ps: [{"params": ps[:3], "weight_decay": 0.05}, {"params": ps[3:], "weight_decay": 0.0}]

    def run(opt, ps, steps):
        for t in steps:
            for g in opt.param_groups:
                g["lr"] = 1e-3 * (1 + t)
            for p, g in zip(ps, grads[t]):
                p.grad = g
            opt.clip_grad_norm_(1.0)
            opt.step()

    full = [p.clone() for p in p0]
    o_full = optim.FusedAdamW(groups(full), betas=BETAS, eps=EPS)
    run(o_full, full, range(2 * k))
    first = [p.clone() for p in p0]
    o1 = optim.FusedAdamW(groups(first), betas=BETAS, eps=EPS)
    run(o1, first, range(k))
    sd = _roundtrip(o1.state_dict())
    steps = [st["step"] for st in sd["state"].values()]
    second = [p.clone() for p in first]
    o2 = optim.FusedAdamW(groups(second), betas=BETAS, eps=EPS)
    o2.load_state_dict(sd)
    run(o2, second, range(k, 2 * k))
    for i, (a, b) in enumerate(zip(second, full)):
        assert torch.equal(a, b), i
        for key in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(o2.state[a][key], o_full.state[b][key]), (i, key)
        assert int(o2.state[a]["step"]) == int(o_full.state[b]["step"]) == 2 * k
    assert len({id(s) for s in steps}) == len(steps) == len(p0)
    assert all(s.dtype == torch.float32 and s.device.type == "cpu" and s.dim() == 0 and float(s) == k for s in steps)


# ------------------------------------------------------------------------------------------ 5. interchange with torch
@pytest.mark.parametrize("direction", ["torch_to_fused", "fused_to_torch"])
def test_state_dict_interchange_with_torch(optim, direction):
    """A torch.optim.AdamW state_dict loaded into FusedAdamW, or a FusedAdamW one (through torch.save / torch.load) loaded into
    torch.optim.AdamW: k steps on one, k on the other, against 2k uninterrupted fp64 steps. Every tensor ends at step 2k, as
    in torch; a step tensor shared between parameters would be advanced once per parameter by torch."""
    k = 3
    gen = torch.Generator(device="cuda").manual_seed(4)
    p0 = _table(gen)
    pair = Pair(optim, [(p0[:3], 0.05), (p0[3:], 0.0)])
    grads = [[_randn(p.shape, gen) for p in p0] for _ in range(2 * k)]
    torch_side = [p.clone() for p in p0]
    o_torch = torch.optim.AdamW([{"params": torch_side[:3], "weight_decay": 0.05}, {"params": torch_side[3:], "weight_decay": 0.0}],
                                betas=BETAS, eps=EPS, foreach=False)
    first, first_ps = (o_torch, torch_side) if direction == "torch_to_fused" else (pair.fused, pair.p32)
    for t in range(2 * k):
        if t == k:
            second_ps = [p.detach().clone() for p in first_ps]
            groups = [{"params": second_ps[:3], "weight_decay": 0.05}, {"params": second_ps[3:], "weight_decay": 0.0}]
            second = (optim.FusedAdamW(groups, betas=BETAS, eps=EPS) if direction == "torch_to_fused" else
                      torch.optim.AdamW(groups, betas=BETAS, eps=EPS, foreach=False))
            second.load_state_dict(_roundtrip(first.state_dict()))
            first, first_ps = second, second_ps
        lr = 1e-3 * (1 + t)
        for g in first.param_groups:
            g["lr"] = lr
        for p, g in zip(first_ps, grads[t]):
            p.grad = g
        torch.nn.utils.clip_grad_norm_(first_ps, 1.0) if isinstance(first, torch.optim.AdamW) else first.clip_grad_norm_(1.0)
        first.step()
        # the fp64 reference alone (Pair.step would also step pair.fused, which may be one of the two above)
        for g in pair.ref.param_groups:
            g["lr"] = lr
        for p, g in zip(pair.p64, grads[t]):
            p.grad = g.double()
        torch.nn.utils.clip_grad_norm_(pair.p64, 1.0, foreach=False)
        pair.ref.step()
        pair.gmax = [max(m, g.abs().max().item()) for m, g in zip(pair.gmax, grads[t])]
        pair.n_steps, pair.lr_sum = pair.n_steps + 1, pair.lr_sum + lr
    pair.check(f"interchange ({direction})", p32=first_ps, state32=first.state)
    assert [float(first.state[p]["step"]) for p in first_ps] == [float(pair.ref.state[p]["step"]) for p in pair.p64] == [2.0 * k] * len(p0)


# ------------------------------------------------------------------------------------------ 6. graph capture
def test_graph_capture_keeps_loaded_state(optim):
    """GraphedTrainStep's warm-up steps the optimizer; afterwards the moments, step counts and weights are bitwise what they
    were before construction (here: state from two eager steps, saved and loaded into the optimizer the graph gets), and
    one replay advances every step count by exactly 1."""
    from egom2p_b200.graphed import GraphedTrainStep
    from test_model_gpu import build_model, to_cuda
    cfg = synth.make_cfg(192, 3, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=512, video_thw=(5, 4, 4))
    n_in = {"tok_cam": [5, 30], "tok_depth": [30, 10], "tok_gaze": [4, 3], "tok_rgb": [25, 21]}
    n_tg = {"tok_cam": [10, 3], "tok_depth": [20, 7], "tok_gaze": [3, 7], "tok_rgb": [15, 18]}
    batches = [to_cuda(synth.make_batch(cfg, B=2, seed=30 + i, n_in=n_in, n_tgt=n_tg)) for i in range(3)]
    model = build_model(cfg).cuda()
    model.load_state_dict(synth.make_state_dict(cfg, 4), strict=True)
    mk = lambda: optim.FusedAdamW([{"params": [p for n, p in model.named_parameters() if "norm" not in n], "weight_decay": 0.05},
                                   {"params": [p for n, p in model.named_parameters() if "norm" in n], "weight_decay": 0.0}],
                                  lr=3e-3, betas=BETAS, eps=EPS)
    eager = mk()
    for md in batches[:2]:
        loss, mod_loss = model(md, 64, 48)
        loss.backward()
        eager.clip_grad_norm_(1.0)
        eager.step()
        eager.zero_grad(set_to_none=True)
    del loss, mod_loss     # a live autograd graph would tie the parameters' AccumulateGrad nodes to this stream during capture
    opt = mk()
    opt.load_state_dict(_roundtrip(eager.state_dict()))
    params = list(model.parameters())
    w0 = [p.detach().clone() for p in params]
    s0 = {p: (opt.state[p]["exp_avg"].clone(), opt.state[p]["exp_avg_sq"].clone(), int(opt.state[p]["step"])) for p in params if opt.state.get(p)}
    assert s0 and all(s == 2 for _, _, s in s0.values())
    runner = GraphedTrainStep(model, opt, batches[2], 64, 48, clip_grad=1.0)
    for p, w in zip(params, w0):
        assert torch.equal(p.detach(), w)
    for p, (m, v, s) in s0.items():
        st = opt.state[p]
        assert torch.equal(st["exp_avg"], m) and torch.equal(st["exp_avg_sq"], v) and int(st["step"]) == s
    runner(batches[0])
    torch.cuda.synchronize()
    assert [int(opt.state[p]["step"]) for p in s0] == [s + 1 for _, _, s in s0.values()]


# ------------------------------------------------------------------------------------------ 7. non-finite norms
@pytest.mark.parametrize("bad", ["nan", "inf"])
def test_non_finite_norm_with_clip(optim, bad):
    """clip_grad_norm_ + step with one non-finite gradient element, as torch does it: a NaN norm gives a NaN coefficient that
    poisons every parameter; an inf norm gives coefficient 0 (and NaN where the gradient is inf, since inf * 0 is NaN)."""
    gen = torch.Generator(device="cuda").manual_seed(5)
    p0 = _table(gen)
    pair = Pair(optim, [(p0[:3], 0.05), (p0[3:], 0.0)])
    grads = [_randn(p.shape, gen) for p in p0]
    pair.step(grads, lrs=[1e-3, 1e-3], max_norm=1.0)
    grads = [_randn(p.shape, gen) for p in p0]
    grads[2][777] = float(bad)
    n32, n64 = pair.step(grads, lrs=[1e-3, 1e-3], max_norm=1.0)
    assert (torch.isnan(n32) if bad == "nan" else torch.isinf(n32)).item() and torch.equal(torch.isnan(n32.cpu()), torch.isnan(n64.cpu()))
    if bad == "nan":
        assert all(torch.isnan(p).all() for p in pair.p64)
    pair.check(f"clip with a {bad} gradient")


@pytest.mark.parametrize("bad", ["nan", "inf"])
def test_scaler_without_clip_reports_norm_only(optim, bad):
    """FusedScalerWithGradNormCount(clip_grad=None) reports the gradient norm but never folds it into the update, also when
    it is inf or NaN (the reference's scaler only computes it then): the step is plain AdamW on the unscaled gradients."""
    gen = torch.Generator(device="cuda").manual_seed(6)
    p0 = [torch.nn.Parameter(p) for p in _table(gen)]
    pair = Pair(optim, [(p0[:3], 0.05), (p0[3:], 0.0)])
    scaler = optim.FusedScalerWithGradNormCount(enabled=False)
    for t in range(2):
        grads = [_randn(p.shape, gen) for p in p0]
        if t == 1:
            grads[4][5] = float(bad)
        for p, g in zip(pair.p64, grads):
            p.grad = g.double()
        norm64 = _norm64(grads)
        loss = sum((p * g).sum() for p, g in zip(p0, grads))
        norm = scaler(loss, pair.fused, clip_grad=None, parameters=p0)
        pair.fused.zero_grad(set_to_none=True)
        pair.ref.step()
        pair.gmax = [max(m, g.abs().nan_to_num(posinf=0.0).max().item()) for m, g in zip(pair.gmax, grads)]
        pair.n_steps, pair.lr_sum = pair.n_steps + 1, pair.lr_sum + 1e-3
        if t == 0:
            assert abs(norm.item() - norm64) <= 1e-5 * norm64
        else:
            assert (torch.isnan(norm) if bad == "nan" else torch.isinf(norm)).item()
    assert not torch.isnan(pair.p64[0]).any()
    pair.check(f"scaler without clip, {bad} gradient")


# ------------------------------------------------------------------------------------------ 8. repeatability of the norm
def test_grad_norm_is_bitwise_repeatable(optim):
    """The norm is a fixed-order sum (per-chunk partials, then one block in a fixed order): twice on the same gradients, and
    in two optimizers over separately allocated copies of the same table, it is bitwise the same. Data-parallel replicas rely
    on this to compute the same clip coefficient. The table has > 1024 chunks, so the finalize loop strides."""
    gen = torch.Generator(device="cuda").manual_seed(7)
    sizes = [(i * 104729) % 400000 + 1 for i in range(1, 65)]
    tables = []
    for _ in range(2):
        tables.append([torch.empty(n, device="cuda") for n in sizes])
    src = [_randn(n, gen) for n in sizes]
    opts = []
    for ps in tables:
        for p, s in zip(ps, src):
            p.grad = s.clone()
        opts.append(optim.FusedAdamW([{"params": ps[::2], "weight_decay": 0.05}, {"params": ps[1::2], "weight_decay": 0.0}]))
    a = opts[0].clip_grad_norm_(1.0).clone()
    b = opts[0].clip_grad_norm_(1.0).clone()
    c = opts[1].clip_grad_norm_(1.0).clone()
    assert opts[0]._n_chunks > 1024
    assert torch.equal(a, b) and torch.equal(a, c), (a.item(), b.item(), c.item())
    torch.testing.assert_close(a.double().cpu(), torch.tensor(_norm64(src), dtype=torch.float64), rtol=1e-5, atol=0)
