"""Whole-step CUDA graph of the training step for small per-GPU batches.

At the reference's own batch size (4 per GPU, cfgs/default/egom2p/models/main/ego-b_mod4_500b_clariden_2048_camcv_depthdenoise.yaml:9)
one step is ~1100 kernel launches of 5-50 us each: issued one at a time from Python the step is bound by the host, not the
GPU (round 1: 33.6 ms / step at b = 4 against ~24 ms of kernel time). `GraphedTrainStep` captures forward + backward +
gradient-norm clip + AdamW (egom2p_b200.optim.FusedAdamW, whose step counts live on the device) ONCE into a CUDA graph and
replays it per step: inputs are copied into static buffers, the loss is read from a static tensor.

What a captured step fixes (checked, not assumed):
  * shapes: batch size, token budgets, and the number of valid target rows of every modality (`static_target_rows`; a batch
    that violates it trips a device-side assertion) -- true for fixed-count masking such as the dense synthetic regime, NOT
    for the reference's Dirichlet-sampled budgets (use the eager path there);
  * the decoder modality order (the reference shuffles it per step with random.sample, egom2p_model.py:312; the loss is
    invariant to it up to summation order, SURVEY.md A7);
  * learning rates / weight decays are read from the optimizer's device table, refreshed by `set_hyper()` between replays.
Single GPU only (DDP's reducer hooks are not captured)."""
from __future__ import annotations

from typing import Dict, Optional

import torch

from .optim import FusedAdamW


class GraphedTrainStep:
    def __init__(self, model, optimizer: FusedAdamW, example_md: Dict[str, Dict[str, torch.Tensor]], num_encoder_tokens: int,
                 num_decoder_tokens: int, clip_grad: Optional[float] = 1.0, loss_type: str = "mod", warmup: int = 3):
        if not isinstance(optimizer, FusedAdamW):
            raise TypeError("GraphedTrainStep needs egom2p_b200.optim.FusedAdamW (device-side step counts)")
        self.model, self.opt = model, optimizer
        self.n_enc, self.n_dec, self.clip, self.loss_type = num_encoder_tokens, num_decoder_tokens, clip_grad, loss_type
        dev = next(model.parameters()).device
        self.static_md = {m: {k: v.to(dev).clone() for k, v in d.items()} for m, d in example_md.items()}

        # ---- shapes the graph bakes in, measured on the example batch (host sync allowed here, before capture)
        info = model.modality_info
        rows = {}
        for m, d in self.static_md.items():
            if m in model.decoder_embeddings:
                rows[m] = int((~d["target_mask"].reshape(d["target_mask"].shape[0], -1)).sum())
        if sum(rows.values()) > num_decoder_tokens * next(iter(self.static_md.values()))["tensor"].shape[0]:
            raise NotImplementedError("GraphedTrainStep: target counts above the decoder budget are truncated per sample; "
                                      "static row counts are only derived for batches that fit the budget")
        import random
        mods = [m for m in self.static_md if m in model.decoder_embeddings]
        model.fixed_decoder_order = random.sample(mods, len(mods))
        model.static_target_rows = rows

        # ---- warm-up on a side stream (allocator, lazy state, cudaFuncSetAttribute), then undo its effect on the weights and on
        # the optimizer state: moments and step counts the optimizer arrived with (e.g. after a resume) are restored, state the
        # warm-up created is left as zero moments at step 0
        params = [p for p in model.parameters() if p.requires_grad]
        backup = [p.detach().clone() for p in params]
        opt_backup = {p: {k: optimizer.state[p][k].detach().clone() for k in ("exp_avg", "exp_avg_sq", "step")}
                      for p in params if "exp_avg" in optimizer.state.get(p, {})}
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(max(1, warmup)):
                self._body()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        with torch.no_grad():
            for p, b in zip(params, backup):
                p.copy_(b)
                st = optimizer.state.get(p)
                if st:
                    for k in ("exp_avg", "exp_avg_sq", "step"):
                        if p in opt_backup:
                            st[k].copy_(opt_backup[p][k])
                        else:
                            st[k].zero_()
        del backup, opt_backup
        model.invalidate_weight_cache()
        optimizer.zero_grad(set_to_none=True)

        # ---- capture
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.mod_loss, self.grad_norm = self._body()
        torch.cuda.synchronize(dev)

    def _body(self):
        self.opt.zero_grad(set_to_none=True)
        loss, mod_loss = self.model(self.static_md, self.n_enc, self.n_dec, loss_type=self.loss_type)
        loss.backward()
        norm = self.opt.clip_grad_norm_(self.clip) if self.clip is not None else None
        self.opt.step()
        return loss.detach(), {m: l.detach() for m, l in mod_loss.items()}, norm

    def set_hyper(self):
        """Re-uploads lr / weight decay from optimizer.param_groups into the device table the captured kernels read (call
        after a scheduler changed them; cheap: 14 KB)."""
        from .optim import _ITEM
        tab = self.opt._stage.numpy().view(_ITEM)
        i = 0
        for p, lr, wd in self.opt._live():
            tab[i]["lr"], tab[i]["wd"] = lr, wd
            i += 1
        self.opt._table.copy_(self.opt._stage, non_blocking=True)

    def __call__(self, md: Dict[str, Dict[str, torch.Tensor]]):
        """One training step on `md` (same shapes as the example batch; host or device tensors). Returns the static loss
        tensor (device); `.mod_loss` / `.grad_norm` hold the other outputs."""
        for m, d in self.static_md.items():
            for k, v in d.items():
                v.copy_(md[m][k], non_blocking=True)
        self.graph.replay()
        return self.loss
