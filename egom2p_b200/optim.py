"""Device-side optimizer tail of the training step (SURVEY.md section 8(f) row 3).

The reference's tail is `NativeScalerWithGradNormCount.__call__` (egom2p/utils/native_scaler.py:27-47): backward,
`clip_grad_norm_(parameters, clip_grad)`, `optimizer.step()` with the AdamW that `create_optimizer` builds
(egom2p/utils/optim_factory.py:157-229: two+ parameter groups, `lr_scale` applied by the scheduler through
`param_group["lr"]`). Here the same two operations run as TWO kernel launches over a device-resident table of all tensors:

  * `FusedAdamW.clip_grad_norm_(max_norm)`  -> egom2p_sumsq_multi: global gradient norm, returned as a device scalar (no
    sync); the clip coefficient is NOT applied to the gradients but folded into
  * `FusedAdamW.step()`                     -> egom2p_adamw_multi_steps: torch.optim.AdamW update of every tensor, reading
    each gradient once as g * min(1, max_norm / (norm + 1e-6)) (NaN when the norm is NaN, as in torch).

`FusedAdamW` is a `torch.optim.Optimizer` (same constructor arguments and param_group keys as `torch.optim.AdamW`, so the
reference's scheduler code that rewrites `param_group["lr"]` / `["weight_decay"]` works unchanged) and
`FusedScalerWithGradNormCount` mirrors the reference scaler's call signature for the bf16 path.

Like torch.optim.AdamW, every tensor has its own step count, and a tensor whose `grad` is None (frozen, or not reached by
the loss) is skipped without counting a step. The counts live in one int32 device array with an entry per live tensor;
each `state[p]["step"]` is a 0-d view of its entry, and the array is rebuilt from those views whenever the set of tensors
with gradients changes. Nothing host-side changes from step to step, so the whole tail can be captured in a CUDA graph
(egom2p_b200/graphed.py). `state_dict()` saves torch's form (an independent float32 CPU `step` per tensor), and
`load_state_dict()` accepts that form from either optimizer."""
from __future__ import annotations

from typing import Iterable, Optional

import numpy as np
import torch

from . import _lib
from .ops import _p, _s, _timed

_ITEM = np.dtype([("p", "<u8"), ("g", "<u8"), ("m", "<u8"), ("v", "<u8"), ("n", "<i8"), ("first_chunk", "<i8"),
                  ("lr", "<f4"), ("wd", "<f4")])
assert _ITEM.itemsize == 56
_CHUNK = 8192


class FusedAdamW(torch.optim.Optimizer):
    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1e-2):
        if lr < 0 or eps < 0 or not 0 <= betas[0] < 1 or not 0 <= betas[1] < 1 or weight_decay < 0:
            raise ValueError("FusedAdamW: invalid hyper-parameter")
        super().__init__(params, dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay))
        b = {tuple(g["betas"]) for g in self.param_groups} | {g["eps"] for g in self.param_groups}
        if len(b) != 2:
            raise NotImplementedError("FusedAdamW: betas / eps must be the same for all parameter groups")
        self._sig = None
        self._table = None
        self._stage = None
        self._n_chunks = 0
        self._n_items = 0
        self._steps: Optional[torch.Tensor] = None      # int32 [n_items]: the step count of every live tensor
        self._steps_key = None                            # ids of the live tensors self._steps was built for
        self._sumsq: Optional[torch.Tensor] = None
        self._pending_clip: Optional[float] = None
        self._partials: Optional[torch.Tensor] = None
        self.bytes_per_step = 0.0

    # ------------------------------------------------------------------ device table
    def _live(self):
        for g in self.param_groups:
            lr, wd = float(g["lr"]), float(g["weight_decay"])
            for p in g["params"]:
                if p.grad is not None:
                    yield p, lr, wd

    def _ensure_table(self):
        live = list(self._live())
        if not live:
            return False
        dev = live[0][0].device
        if self._sumsq is None:
            self._sumsq = torch.zeros(1, dtype=torch.float32, device=dev)
        key = tuple(id(p) for p, _, _ in live)
        if key != self._steps_key:
            self._bind_steps([p for p, _, _ in live], dev)
            self._steps_key = key
        sig = tuple((p.data_ptr(), p.grad.data_ptr(), lr, wd) for p, lr, wd in live)
        if sig == self._sig:
            return True
        tab = np.zeros(len(live), dtype=_ITEM)
        chunk = 0
        nbytes = 0
        for i, (p, lr, wd) in enumerate(live):
            if p.dtype != torch.float32 or p.grad.dtype != torch.float32 or not p.is_contiguous() or not p.grad.is_contiguous():
                raise TypeError("FusedAdamW: parameters and gradients must be contiguous fp32 CUDA tensors")
            st = self.state[p]
            n = p.numel()
            tab[i] = (p.data_ptr(), p.grad.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), n, chunk, lr, wd)
            chunk += (n + _CHUNK - 1) // _CHUNK
            nbytes += n
        raw = torch.from_numpy(tab.view(np.uint8).reshape(-1))
        if self._stage is None or self._stage.numel() != raw.numel():
            self._stage = torch.empty(raw.numel(), dtype=torch.uint8).pin_memory()
            self._table = torch.empty(raw.numel(), dtype=torch.uint8, device=dev)
        self._stage.copy_(raw)
        self._table.copy_(self._stage, non_blocking=True)
        self._sig, self._n_items, self._n_chunks = sig, len(live), chunk
        if self._partials is None or self._partials.numel() < chunk:
            self._partials = torch.empty(chunk, dtype=torch.float32, device=dev)
        self.bytes_per_step = nbytes * 28.0
        self._grad_bytes = nbytes * 4.0
        return True

    def _bind_steps(self, params, dev):
        """Builds the step array for `params` (the live tensors, in table order) and points each state["step"] at its entry.
        A tensor keeps the count it has (a view into the previous array, or a loaded value); a tensor without state starts
        with zero moments and step 0. Runs when the set of live tensors changes, not per step."""
        for p in params:
            st = self.state[p]
            if "exp_avg" not in st:
                st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["step"] = torch.zeros((), dtype=torch.int32, device=dev)
        self._steps = torch.stack([self.state[p]["step"].detach().reshape(()).to(device=dev, dtype=torch.int32) for p in params])
        for i, p in enumerate(params):
            self.state[p]["step"] = self._steps[i]

    def state_dict(self):
        """torch.optim.AdamW's form: every tensor's state holds its own float32 CPU `step`, so that torch.load does not
        hand one shared tensor to every parameter (torch.optim.AdamW would then advance it once per parameter)."""
        sd = super().state_dict()
        state = {k: dict(st) for k, st in sd["state"].items()}
        keys = [k for k, st in state.items() if "step" in st]
        if keys:
            steps = [state[k]["step"].detach().reshape(()) for k in keys]
            vals = torch.stack([s.to(device=steps[0].device, dtype=torch.float32) for s in steps]).cpu()
            for i, k in enumerate(keys):
                state[k]["step"] = vals[i].clone()
        sd["state"] = state
        return sd

    def load_state_dict(self, state_dict):
        """Accepts a state_dict of this class or of torch.optim.AdamW (per-tensor `step`, float or int, CPU or device)."""
        for g in state_dict["param_groups"]:
            if g.get("amsgrad") or g.get("maximize") or g.get("decoupled_weight_decay", True) is False:
                raise NotImplementedError("FusedAdamW: amsgrad, maximize and coupled (Adam) weight decay are not supported")
        super().load_state_dict(state_dict)
        self._steps_key = self._sig = None     # new moment tensors and step counts: rebuild the table and the step array

    # ------------------------------------------------------------------ public API
    @torch.no_grad()
    def grad_norm(self) -> torch.Tensor:
        """Global 2-norm of all gradients of this optimizer's parameters as a device scalar (no host sync), computed in one
        launch. It does not affect the next `step()`."""
        if not self._ensure_table():
            return torch.zeros(())
        lib = _lib.load()
        with _timed("optimizer", self._grad_bytes, "byte"):
            _lib.check(lib.egom2p_sumsq_multi(_p(self._table), self._n_items, self._n_chunks, _p(self._partials), _p(self._sumsq), _s()),
                       "sumsq_multi")
        return self._sumsq.sqrt().reshape(())

    @torch.no_grad()
    def clip_grad_norm_(self, max_norm: float) -> torch.Tensor:
        """`grad_norm()`, with the clip applied inside the next `step()` (torch.nn.utils.clip_grad_norm_ semantics: gradients
        are scaled by min(1, max_norm / (norm + 1e-6)), NaN for a NaN norm -- here on the fly instead of in place)."""
        norm = self.grad_norm()
        self._pending_clip = float(max_norm)
        return norm

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        clip = self._pending_clip
        self._pending_clip = None
        if not self._ensure_table():
            return loss
        lib = _lib.load()
        g0 = self.param_groups[0]
        with _timed("optimizer", self.bytes_per_step, "byte"):
            _lib.check(lib.egom2p_adamw_multi_steps(_p(self._table), self._n_items, self._n_chunks, float(g0["betas"][0]),
                                                    float(g0["betas"][1]), float(g0["eps"]), _p(self._steps),
                                                    _p(self._sumsq) if clip is not None else None, clip if clip is not None else 0.0,
                                                    _s()), "adamw_multi_steps")
        return loss


class FusedScalerWithGradNormCount:
    """Call-compatible stand-in for egom2p/utils/native_scaler.py:NativeScalerWithGradNormCount on the bf16 path (where
    the reference's GradScaler is disabled and the object only sequences backward / clip / step)."""
    state_dict_key = "amp_scaler"

    def __init__(self, enabled: bool = False):
        if enabled:
            raise NotImplementedError("loss scaling (fp16) is not part of the bf16 ego-b path")

    def __call__(self, loss, optimizer, clip_grad=None, skip_grad=None, parameters: Optional[Iterable] = None, create_graph=False,
                 update_grad=True, compute_grad_norm=True):
        loss.backward(create_graph=create_graph)
        if not update_grad:
            return None
        if skip_grad is not None:
            raise NotImplementedError("skip_grad needs a host decision per step; use clip_grad")
        fused = isinstance(optimizer, FusedAdamW)
        norm = None
        if clip_grad is not None:
            norm = optimizer.clip_grad_norm_(clip_grad) if fused else torch.nn.utils.clip_grad_norm_(parameters, clip_grad)
        elif compute_grad_norm and fused:   # reported only: the reference's get_grad_norm_ leaves the gradients as they are
            norm = optimizer.grad_norm()
        optimizer.step()
        return norm

    def state_dict(self):
        return {}

    def load_state_dict(self, state_dict):
        pass
