"""GPU: several optimizer steps of the training loop body (forward + backward + clip_grad_norm_(1.0) + fused AdamW,
run_training_egom2p.py:701-746) against the same loop over the CPU oracle. Guards the bf16 operand cache of the module:
every step must run on the weights the optimizer just wrote, so the loss trajectory has to follow the oracle's
(a stale cache shows up from step 2 on; the learning rate is large so that one update moves the loss visibly)."""
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

import egom2p_oracle as orc  # noqa: E402
import synth  # noqa: E402
from test_model_gpu import build_model, to_cuda  # noqa: E402

STEPS = 4
LR = 3e-3


def _oracle_losses(sd, cfg, md, n_enc, n_dec, orders):
    leaf = {}
    for k, v in sd.items():
        if k.endswith("to_logits.weight") or (k.startswith("decoder_embeddings") and k.endswith("mod_emb")):
            continue
        leaf[k] = v.clone().requires_grad_(v.is_floating_point() and not k.endswith("pos_emb")
                                           and not (k.endswith(".bias") and "proj_context" not in k))
    for m in cfg["mods"]:
        leaf[f"decoder_embeddings.{m}.to_logits.weight"] = leaf[f"decoder_embeddings.{m}.token_emb.weight"]
        leaf[f"decoder_embeddings.{m}.mod_emb"] = leaf[f"encoder_embeddings.{m}.mod_emb"]
    params = list({id(t): t for t in leaf.values() if t.requires_grad}.values())
    opt = torch.optim.AdamW(params, lr=LR, betas=(0.9, 0.95), weight_decay=0.05)
    losses = []
    for order in orders:
        out = orc.forward(leaf, cfg, md, n_enc, n_dec, dec_order=order, loss_type="mod")
        out["loss"].backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
        losses.append(out["loss"].item())
    return losses


def test_loss_trajectory_follows_oracle():
    cfg = synth.make_cfg(192, 3, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=512, video_thw=(5, 4, 4))
    md = synth.make_batch(cfg, B=4, seed=11,
                          n_in={"tok_cam": [5, 0, 30, 2], "tok_depth": [30, 10, 0, 1], "tok_gaze": [4, 0, 30, 0], "tok_rgb": [25, 40, 4, 0]},
                          n_tgt={"tok_cam": [10, 30, 0, 1], "tok_depth": [20, 0, 40, 0], "tok_gaze": [3, 0, 0, 0], "tok_rgb": [15, 18, 70, 0]})
    sd = synth.make_state_dict(cfg, 5)
    mods = list(cfg["mods"])
    orders = []
    for s in range(STEPS):
        random.seed(100 + s)
        orders.append(random.sample(mods, len(mods)))
    ref = _oracle_losses(sd, cfg, md, 64, 48, orders)

    model = build_model(cfg).cuda()
    model.load_state_dict(sd, strict=True)
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=LR, betas=(0.9, 0.95), weight_decay=0.05, fused=True)
    mdc = to_cuda(md)
    got = []
    for s in range(STEPS):
        random.seed(100 + s)
        loss, _ = model(mdc, 64, 48, loss_type="mod")
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
        got.append(loss.item())
    assert ref[0] - ref[-1] > 0.05 * ref[0], f"oracle loss did not move enough for the test to discriminate: {ref}"
    for s, (a, b) in enumerate(zip(got, ref)):
        tol = 1e-3 if s == 0 else 1.5e-2   # later steps compound bf16-vs-fp32 update differences; a stale cache is ~15 % off
        assert abs(a - b) / abs(b) < tol, f"step {s}: loss {a} vs oracle {b}\nours {got}\noracle {ref}"

    # the cached bf16 operands are exactly the rounded masters after the last update, once the next forward refreshes them
    with torch.no_grad():
        random.seed(0)
        model(mdc, 64, 48, loss_type="mod")
    blk = model.encoder[0]
    wq = model._wcache[("e", 0, "qkv")][3]
    assert torch.equal(wq, blk.attn.qkv.weight.detach().to(torch.bfloat16))
    w2 = model._wcache[("e", 0, "w2")][3]
    F = blk.mlp.fc2.weight.shape[1]
    assert torch.equal(w2[:, :F], blk.mlp.fc2.weight.detach().to(torch.bfloat16))
    w13 = model._wcache[("e", 0, "w13")][3]
    v = w13.view(-1, 2, 32, w13.shape[1])
    Fh = blk.mlp.fc1.weight.shape[0]
    assert torch.equal(v[:, 0].reshape(-1, w13.shape[1])[:Fh], blk.mlp.fc1.weight.detach().to(torch.bfloat16))
    assert torch.equal(v[:, 1].reshape(-1, w13.shape[1])[:Fh], blk.mlp.fc3.weight.detach().to(torch.bfloat16))


def test_loop_body_under_autocast_and_scaler():
    """The reference calls the model under torch.cuda.amp.autocast(bfloat16) and steps through its GradScaler wrapper with
    the scaler disabled for bf16 (run_training_egom2p.py:518,725-746; native_scaler.py:27-47). The module computes with its
    own kernels, so that context must change nothing: same losses as the plain loop (fp32 atomics in dQ / embedding
    gradients make later steps differ in the last bits only)."""
    cfg = synth.make_cfg(192, 3, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=512, video_thw=(5, 4, 4))
    md = synth.make_batch(cfg, B=4, seed=12,
                          n_in={"tok_cam": [5, 0, 30, 2], "tok_depth": [30, 10, 0, 1], "tok_gaze": [4, 0, 30, 0], "tok_rgb": [25, 40, 4, 0]},
                          n_tgt={"tok_cam": [10, 30, 0, 1], "tok_depth": [20, 0, 40, 0], "tok_gaze": [3, 0, 0, 0], "tok_rgb": [15, 18, 70, 0]})
    sd = synth.make_state_dict(cfg, 6)
    mdc = to_cuda(md)

    def loop(amp):
        model = build_model(cfg).cuda()
        model.load_state_dict(sd, strict=True)
        params = [p for p in model.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=LR, betas=(0.9, 0.95), weight_decay=0.05, fused=True)
        scaler = torch.amp.GradScaler("cuda", enabled=False)
        out = []
        for s in range(3):
            random.seed(200 + s)
            if amp:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    loss, mod_loss = model({m: dict(d) for m, d in mdc.items()}, 64, 48, loss_type="mod")
                assert loss.dtype == torch.float32 and all(v.dtype == torch.float32 for v in mod_loss.values())
                scaler.scale(loss).backward()
                scaler.unscale_(opt)
                torch.nn.utils.clip_grad_norm_(params, 1.0)
                scaler.step(opt)
                scaler.update()
            else:
                loss, _ = model({m: dict(d) for m, d in mdc.items()}, 64, 48, loss_type="mod")
                loss.backward()
                torch.nn.utils.clip_grad_norm_(params, 1.0)
                opt.step()
            opt.zero_grad(set_to_none=True)
            out.append(loss.item())
        return out

    plain, amp = loop(False), loop(True)
    assert plain[0] == amp[0], (plain, amp)
    for a, b in zip(plain, amp):
        assert abs(a - b) <= 2e-4 * abs(a), (plain, amp)
    assert plain[-1] < 0.95 * plain[0]


def test_graphed_step_matches_eager_per_tensor_steps():
    """egom2p_b200.graphed.GraphedTrainStep (whole-step CUDA graph: forward + backward + clip + FusedAdamW) reproduces the
    eager step: same losses and the same weights after 3 steps on 3 different batches with equal target counts."""
    import copy
    from egom2p_b200.graphed import GraphedTrainStep
    from egom2p_b200.optim import FusedAdamW
    from test_model_gpu import build_model, to_cuda
    cfg = synth.make_cfg(192, 3, 2, 2, ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"], video_vocab=512, video_thw=(5, 4, 4))
    n_in = {"tok_cam": [5, 30], "tok_depth": [30, 10], "tok_gaze": [4, 3], "tok_rgb": [25, 21]}
    n_tg = {"tok_cam": [10, 3], "tok_depth": [20, 7], "tok_gaze": [3, 7], "tok_rgb": [15, 18]}
    batches = [to_cuda(synth.make_batch(cfg, B=2, seed=30 + i, n_in=n_in, n_tgt=n_tg)) for i in range(4)]
    sd = synth.make_state_dict(cfg, 4)
    models = []
    for _ in range(2):
        m = build_model(cfg).cuda()
        m.load_state_dict(sd, strict=True)
        models.append(m)
    eager, graphed = models
    mk = lambda m: FusedAdamW([{"params": [p for n, p in m.named_parameters() if "norm" not in n], "weight_decay": 0.05},
                               {"params": [p for n, p in m.named_parameters() if "norm" in n], "weight_decay": 0.0}],
                              lr=3e-3, betas=(0.9, 0.95), eps=1e-8)
    o_e, o_g = mk(eager), mk(graphed)
    runner = GraphedTrainStep(graphed, o_g, batches[3], 64, 48, clip_grad=1.0)
    eager.fixed_decoder_order = list(graphed.fixed_decoder_order)
    for i in range(3):
        if i == 2:   # a scheduler changes the learning rate between steps
            for g1, g2 in zip(o_e.param_groups, o_g.param_groups):
                g1["lr"] = g2["lr"] = 1e-3
            runner.set_hyper()
        loss_e, _ = eager(batches[i], 64, 48)
        loss_e.backward()
        n_e = o_e.clip_grad_norm_(1.0)
        o_e.step()
        o_e.zero_grad(set_to_none=True)
        loss_g = runner(batches[i])
        torch.cuda.synchronize()
        assert abs(loss_e.item() - loss_g.item()) <= 2e-4 * abs(loss_e.item()), (i, loss_e.item(), loss_g.item())
        assert abs(n_e.item() - runner.grad_norm.item()) <= 2e-3 * n_e.item()
    steps = [int(st["step"]) for st in o_g.state.values() if st]
    assert steps and steps == [3] * len(steps), steps
    # Adam moves every element by about +-lr per step whatever the gradient's size, and dQ accumulates through fp32 atomics
    # (run-to-run noise in the last bits): elements with a near-zero gradient may step in opposite directions in the two runs.
    # So: the bulk of the weights agrees closely, and no element is further apart than the steps taken (3e-3 + 3e-3 + 1e-3).
    lr_sum = 7e-3
    for a, b in zip(graphed.parameters(), eager.parameters()):
        d = (a.detach() - b.detach()).abs()
        assert d.max().item() <= 2.2 * lr_sum and d.mean().item() <= 0.05 * lr_sum, (tuple(a.shape), d.max().item(), d.mean().item())
