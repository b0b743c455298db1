"""``FusedAdam`` -- torch.optim.Adam semantics (torch/optim/adam.py single-tensor path, as driven by
ps_vae/lightning.py:204-205) in ONE vectorised CUDA pass per contiguous parameter range (28 B/param).

It is a real ``torch.optim.Optimizer``: ``param_groups`` / ``state_dict()`` / ``load_state_dict()`` keep torch's
layout (``state[p] = {'step', 'exp_avg', 'exp_avg_sq'}``), so ``CosineAnnealingLR`` and Lightning checkpointing
work unchanged.  ``exp_avg`` / ``exp_avg_sq`` are views into flat moment buffers that mirror the parameter
arena; gradients are consumed straight from the arena's flat gradient buffer (after a data-parallel
all-reduce they hold the SUM over ranks: ``grad_scale = 1 / world_size`` folds the averaging into the pass).
In bf16 mode the same pass also refreshes the bf16 operand copy the tcgen05 GEMMs read.

``amsgrad`` (state key ``max_exp_avg_sq``, a third flat buffer) and ``maximize`` -- both reachable through
``Adam(self.parameters(), **self.hparams["optimizer"])`` -- take the general form of the kernel (one element per thread);
``capturable`` / ``differentiable`` are not on the reference's path and raise.  Every update goes through ``psvae_adam_step_clip``.

Gradient clipping (Lightning's ``gradient_clip_val`` / ``gradient_clip_algorithm``) happens inside the same pass when ``clip_mode`` is set
(``DataParallelTrainer`` sets it, as it sets ``grad_scale``): ``"norm"`` scales ``g`` by ``grad_scale * clip_coef`` (``clip_coef``: a device
scalar written by ``psvae_grad_norm``), ``"value"`` clamps ``g * grad_scale`` at ``clip_value`` -- before weight decay and maximize, where
torch clips.  The ``.grad``
tensors themselves are not rewritten.
"""
from __future__ import annotations

from typing import Iterable, List, Optional, Tuple

import torch

from . import _lib as L
from .engine import ParamArena, _on, _stream_ptr


class FusedAdam(torch.optim.Optimizer):
    def __init__(self, params: Iterable, lr: float = 1e-3, betas: Tuple[float, float] = (0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0, amsgrad: bool = False, *, arena: Optional[ParamArena] = None, maximize: bool = False,
                 foreach=None, capturable: bool = False, differentiable: bool = False, fused=None):
        if capturable or differentiable:
            raise NotImplementedError("FusedAdam implements eager torch.optim.Adam (no capturable / differentiable)")
        if lr < 0.0:
            raise ValueError(f"Invalid learning rate: {lr}")
        if eps < 0.0:
            raise ValueError(f"Invalid epsilon value: {eps}")
        if not 0.0 <= betas[0] < 1.0:
            raise ValueError(f"Invalid beta parameter at index 0: {betas[0]}")
        if not 0.0 <= betas[1] < 1.0:
            raise ValueError(f"Invalid beta parameter at index 1: {betas[1]}")
        if weight_decay < 0.0:
            raise ValueError(f"Invalid weight_decay value: {weight_decay}")
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=bool(amsgrad), maximize=bool(maximize), foreach=None,
                        capturable=False, differentiable=False, fused=None)
        super().__init__(params, defaults)
        if arena is None:
            raise ValueError("FusedAdam needs the parameter arena (use PseudoSpeakerVAE.configure_optimizers or HotPath.arena)")
        self.arena = arena
        self.grad_scale = 1.0          # 1 / world_size after a SUM all-reduce
        self.clip_mode = "none"        # "none" | "norm" (g * (grad_scale * clip_coef)) | "value" (clamp(g * grad_scale, -clip_value, clip_value))
        self.clip_coef: Optional[torch.Tensor] = None   # device fp32 scalar written by psvae_grad_norm
        self.clip_value = 0.0
        self._m: Optional[torch.Tensor] = None
        self._v: Optional[torch.Tensor] = None
        self._vmax: Optional[torch.Tensor] = None      # amsgrad: running maximum of exp_avg_sq
        self._offsets = {id(p): off for p, off in arena.entries}
        for g in self.param_groups:
            for p in g["params"]:
                if id(p) not in self._offsets:
                    raise ValueError("FusedAdam can only optimise parameters that live in the arena")

    # ---- flat moment buffers ----------------------------------------------------------------------
    def _moments(self) -> Tuple[torch.Tensor, torch.Tensor]:
        flat = self.arena.ensure()
        if self._m is None or self._m.device != flat.device:
            old_m, old_v = self._m, self._v
            old_x = self._vmax
            self._m = torch.zeros_like(flat)
            self._v = torch.zeros_like(flat)
            if any(g["amsgrad"] for g in self.param_groups):
                self._vmax = torch.zeros_like(flat)
            if old_m is not None:
                self._m.copy_(old_m)
                self._v.copy_(old_v)
                if old_x is not None and self._vmax is not None:
                    self._vmax.copy_(old_x)
            self._bind_state()
        return self._m, self._v

    def _bind_state(self) -> None:
        """Point state[p]['exp_avg'/'exp_avg_sq'] at views of the flat buffers (keeping any loaded values)."""
        for g in self.param_groups:
            for p in g["params"]:
                off, n = self._offsets[id(p)], p.numel()
                st = self.state[p]
                mv, vv = self._m[off:off + n].view(p.shape), self._v[off:off + n].view(p.shape)
                if "exp_avg" in st and st["exp_avg"].data_ptr() != mv.data_ptr():
                    mv.copy_(st["exp_avg"])
                    vv.copy_(st["exp_avg_sq"])
                st["exp_avg"], st["exp_avg_sq"] = mv, vv
                if g["amsgrad"] and self._vmax is not None:
                    xv = self._vmax[off:off + n].view(p.shape)
                    if "max_exp_avg_sq" in st and st["max_exp_avg_sq"].data_ptr() != xv.data_ptr():
                        xv.copy_(st["max_exp_avg_sq"])
                    st["max_exp_avg_sq"] = xv
            # one shared CPU step counter per group (torch keeps one per parameter; they always agree here)
            vals = {float(self.state[p]["step"]) for p in g["params"] if "step" in self.state[p]}
            if len(vals) > 1:
                raise RuntimeError("FusedAdam expects all parameters of a group to share one step count")
            shared = torch.tensor(vals.pop() if vals else 0.0, dtype=torch.float32)
            for p in g["params"]:
                self.state[p]["step"] = shared

    def load_state_dict(self, state_dict) -> None:
        super().load_state_dict(state_dict)
        if self._m is not None:
            self._bind_state()

    # ---- ranges -----------------------------------------------------------------------------------
    def _ranges(self, spans: List[Tuple[int, int]]) -> List[Tuple[int, int]]:
        """Merge [offset, end) spans whose gap holds nothing but arena padding (zero-valued, zero-gradient).  A gap in which a
        parameter lives that is NOT being updated (frozen, or without a gradient this step) is never bridged."""
        owned = sorted(off for _, off in self.arena.entries)
        out: List[List[int]] = []
        for a, b in sorted(spans):
            if out and a - out[-1][1] < 64 and not any(out[-1][1] <= o < a for o in owned):
                out[-1][1] = max(out[-1][1], b)
            else:
                out.append([a, b])
        return [(a, b) for a, b in out]

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        self._update()
        return loss

    def _update(self, counters: Optional[torch.Tensor] = None, lrs: Optional[torch.Tensor] = None) -> None:
        """The update of every group with gradients, one pass per merged span.  ``counters`` / ``lrs``: the device-counter form a CUDA graph
        of the train step replays (graphs.py) -- one ``psvae_step_counters`` block per group (int64 [groups, COUNTER_SLOTS]) and one fp64
        learning rate per group, read on the device.  That form moves no host state: the caller advances the step
        counts, the arena epoch and the shadow mark, and the device block, itself."""
        dc = counters is not None
        clip = {"none": L.CLIP_NONE, "norm": L.CLIP_NORM, "value": L.CLIP_VALUE}[self.clip_mode]
        if clip == L.CLIP_NORM and (self.clip_coef is None or self.clip_coef.dtype != torch.float32):
            raise ValueError("clip_mode 'norm' needs clip_coef, a device fp32 scalar")
        flat = self.arena.ensure()
        dev = flat.device
        if dev.type != "cuda":
            raise RuntimeError("FusedAdam runs on a CUDA (B200) device only; there is no CPU fallback")
        m, v = self._moments()
        gflat = self.arena.flat_grad()
        lib = L.lib()
        stream = _stream_ptr(dev)
        touched = False
        # every span below also rewrites its slice of the bf16 copy: a copy that was current stays current whatever the update covers
        shadow_was_current = not dc and self.arena.shadow_current()
        for gi, group in enumerate(self.param_groups):
            with_grad = [p for p in group["params"] if p.grad is not None]
            if not with_grad:
                continue
            if gflat is None:
                if dc:
                    raise NotImplementedError("the device-counter update reads the gradients from the arena's flat gradient buffer")
                # gradients were produced outside the fused step (plain autograd on a caller's own loss): gather them
                gflat = self.arena.stage_buffer()
                gflat.zero_()          # padding between merged spans must read as zero gradient
                for p in with_grad:
                    off = self._offsets[id(p)]
                    gflat[off:off + p.numel()].copy_(p.grad.reshape(-1))
            step_t = self.state[with_grad[0]]["step"]
            step = 0 if dc else int(step_t.item()) + 1
            beta1, beta2 = group["betas"]
            spans = [(self._offsets[id(p)], self._offsets[id(p)] + p.numel()) for p in with_grad]
            for a, b in self._ranges(spans):
                shadow = None
                if self.arena.shadow is not None and self.arena.shadow.device == dev:
                    shadow = self.arena.shadow.data_ptr() + 2 * a
                vmax = self._vmax.data_ptr() + 4 * a if group["amsgrad"] else None
                with _on(dev):
                    rc = lib.psvae_adam_step_clip(flat.data_ptr() + 4 * a, gflat.data_ptr() + 4 * a, m.data_ptr() + 4 * a, v.data_ptr() + 4 * a, vmax,
                                                  b - a, float(group["lr"]), step, L.ptr(lrs[gi]) if dc else None,
                                                  counters[gi].data_ptr() if dc else None, float(beta1), float(beta2), float(group["eps"]),
                                                  float(group["weight_decay"]), float(self.grad_scale), int(bool(group["amsgrad"])),
                                                  int(bool(group["maximize"])), clip, L.ptr(self.clip_coef), float(self.clip_value), shadow, stream)
                L.check(rc, "psvae_adam_step_clip")
                touched = True
            if not dc:
                step_t += 1
        if touched and not dc:
            self.arena.epoch += 1
            if self.arena.shadow is not None and (self.covers_arena() or shadow_was_current):
                self.arena.mark_shadow_current()

    def covers_arena(self) -> bool:
        """Does one update rewrite every parameter of the arena (so that it also leaves the whole bf16 copy current)?"""
        return all(p.grad is not None for g in self.param_groups for p in g["params"]) and \
            sum(len(g["params"]) for g in self.param_groups) == len(self.arena.entries)
