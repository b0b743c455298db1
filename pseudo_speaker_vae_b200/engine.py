"""Host side of the hot path: flat parameter arena + the calls into the C-ABI.

The reference keeps 18 (+2..6) separate ``nn.Parameter`` tensors and lets autograd / ``torch.optim.Adam`` /
DDP walk them (ps_vae/lightning.py:204-205, ps_vae/training.py:78).  Here every parameter of the VAE and of
the latent classifier is a *view* into one flat fp32 buffer whose layout ``psvae_model_desc_init`` defines,
with sibling flat buffers for the gradients (and, in optim.py, Adam's moments).  State-dict keys, shapes and
values are unchanged -- the modules still own ordinary ``nn.Parameter`` objects -- but the fused train step,
the Adam update and the data-parallel all-reduce each become one pass over one buffer.

``HotPath`` is the object the drop-in modules (model.py, lightning.py, inference.py) delegate to.
"""
from __future__ import annotations

import copy
import ctypes as C
import weakref
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import _lib as L

PRECISIONS = {"fp32": L.FP32, "float32": L.FP32, "32": L.FP32, "highest": L.FP32,
              "bf16": L.BF16, "bfloat16": L.BF16, "medium": L.BF16, "bf16-mixed": L.BF16}


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _on(device: torch.device):
    """Device guard for a library call: the library launches on the CURRENT device (cudaGetDevice), so a module on cuda:1 must make
    cuda:1 current for the duration of the call whatever the caller's current device is."""
    return torch.cuda.device(device)


class _Token:
    """Marks a staging buffer as owned by a loss whose backward has not run yet (weakly held by the arena)."""

    __slots__ = ("buf", "__weakref__")

    def __init__(self, buf: torch.Tensor):
        self.buf = buf


class ParamArena:
    """One flat fp32 buffer holding every parameter; the modules' ``nn.Parameter``s are views into it."""

    def __init__(self, desc: L.ModelDesc, entries: Sequence[Tuple[nn.Parameter, int]]):
        self.desc = desc
        self.entries: List[Tuple[nn.Parameter, int]] = list(entries)
        self.numel = int(desc.total_numel)
        self.flat: Optional[torch.Tensor] = None
        self._gbuf: List[torch.Tensor] = []                      # gradient staging buffers (see stage_buffer); two in steady state
        self._inflight: "weakref.WeakSet[_Token]" = weakref.WeakSet()
        self.shadow: Optional[torch.Tensor] = None               # bf16 operand copy for the tcgen05 engine
        self._shadow_versions: Optional[Tuple[int, ...]] = None
        self._shadow_epoch = -1
        self.epoch = 0    # bumped whenever the library itself rewrites the parameters (fused Adam)
        self._attach(self.entries[0][0].device)

    # ---- layout ---------------------------------------------------------------------------------
    def _attach(self, device: torch.device) -> None:
        flat = torch.zeros(self.numel, dtype=torch.float32, device=device)
        with torch.no_grad():
            for p, off in self.entries:
                n = p.numel()
                flat[off:off + n].copy_(p.detach().reshape(-1).to(device=device, dtype=torch.float32))
                p.data = flat[off:off + n].view(p.shape)
        self.flat = flat
        self._gbuf = []
        self.shadow = None
        self._shadow_versions = None

    # transient state (staging buffers, the bf16 operand copy, ownership tokens) is per instance and rebuilt on demand: it is neither
    # pickled (torch.save(module)) nor deep-copied (SWA / EMA callbacks, ddp_spawn)
    def __getstate__(self):
        st = dict(self.__dict__)
        st.update(_gbuf=[], _inflight=None, shadow=None, _shadow_versions=None, _shadow_epoch=-1)
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        self._inflight = weakref.WeakSet()

    def attached(self) -> bool:
        base = self.flat.data_ptr()
        dev = self.flat.device
        for p, off in self.entries:
            if p.device != dev or p.dtype != torch.float32 or p.data_ptr() != base + 4 * off or not p.is_contiguous():
                return False
        return True

    def ensure(self) -> torch.Tensor:
        """(Re)build the arena if a ``.to()`` / ``.double()`` / foreign optimiser moved the parameters out of it."""
        if not self.attached():
            p0 = self.entries[0][0]
            if p0.dtype != torch.float32:
                raise TypeError(f"pseudo_speaker_vae_b200 kernels run on float32 parameters, got {p0.dtype}")
            self._attach(p0.device)
        return self.flat

    @property
    def device(self) -> torch.device:
        return self.entries[0][0].device

    # ---- gradients ------------------------------------------------------------------------------
    def stage_buffer(self) -> torch.Tensor:
        """A flat gradient buffer that no live ``p.grad`` aliases (gradient accumulation keeps that one alive) and that no
        loss whose ``backward()`` is still to come owns (two ``training_step`` calls before one backward each get their own)."""
        dev = self.ensure().device       # the arena follows the parameters first (a module moved with .to() re-attaches here, not on the CPU copy)
        self._gbuf = [g for g in self._gbuf if g.device == dev]
        live = {p.grad.data_ptr() for p, _ in self.entries if p.grad is not None}
        busy = [t.buf for t in self._inflight]
        for g in self._gbuf:
            lo, hi = g.data_ptr(), g.data_ptr() + 4 * self.numel
            if any(lo <= q < hi for q in live) or any(b is g for b in busy):
                continue
            return g
        g = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        self._gbuf.append(g)
        return g

    def own(self, gflat: torch.Tensor) -> _Token:
        tok = _Token(gflat)
        self._inflight.add(tok)
        return tok

    def grad_views(self, gflat: torch.Tensor) -> List[torch.Tensor]:
        return [gflat[off:off + p.numel()].view(p.shape) for p, off in self.entries]

    def flat_grad(self) -> Optional[torch.Tensor]:
        """The flat buffer the current ``.grad`` tensors live in (None if they do not all alias one buffer)."""
        for g in self._gbuf:
            base = g.data_ptr()
            ok = True
            for p, off in self.entries:
                if p.requires_grad and (p.grad is None or p.grad.data_ptr() != base + 4 * off):
                    ok = False
                    break
            if ok:
                return g
        return None

    # ---- bf16 operand copy ----------------------------------------------------------------------
    def shadow_ptr(self, desc_ref) -> int:
        self.ensure()
        versions = tuple(p._version for p, _ in self.entries)
        if self.shadow is None or self.shadow.device != self.flat.device or versions != self._shadow_versions or self._shadow_epoch != self.epoch:
            if self.shadow is None or self.shadow.device != self.flat.device:
                self.shadow = torch.empty(self.numel, dtype=torch.bfloat16, device=self.flat.device)
            with _on(self.flat.device):
                L.check(L.lib().psvae_refresh_shadow(desc_ref, self.flat.data_ptr(), self.shadow.data_ptr(), _stream_ptr(self.flat.device)),
                        "psvae_refresh_shadow")
            self._shadow_versions = versions
            self._shadow_epoch = self.epoch
        return self.shadow.data_ptr()

    def shadow_current(self) -> bool:
        """Is the bf16 copy on the arena's device and up to date with the parameters (nothing rewrote them since it was last written)?"""
        return self.shadow is not None and self.shadow.device == self.flat.device and self._shadow_epoch == self.epoch \
            and self._shadow_versions == tuple(p._version for p, _ in self.entries)

    def mark_shadow_current(self) -> None:
        """Called by the fused Adam, which writes the bf16 copy itself."""
        self._shadow_versions = tuple(p._version for p, _ in self.entries)
        self._shadow_epoch = self.epoch


class _FusedLoss(torch.autograd.Function):
    """Gives ``loss.backward()`` its meaning: the gradients were already computed by the fused kernel call."""

    @staticmethod
    def forward(ctx, loss_value: torch.Tensor, gflat: torch.Tensor, arena: ParamArena, *params):
        ctx.arena = arena
        ctx.gflat = gflat
        ctx.token = arena.own(gflat)      # the staging buffer is this loss's until its backward has run (or the loss is dropped)
        ctx.needs = [p.requires_grad for p in params]
        return loss_value.clone()

    @staticmethod
    def backward(ctx, gout):
        g = ctx.gflat
        if g is None:
            raise RuntimeError("the fused gradients of this loss were already handed to autograd (backward through the same training_step "
                               "output twice); call training_step again")
        ctx.gflat = ctx.token = None
        g.mul_(gout)     # d(total)/d(loss); a ones tensor for a plain loss.backward()
        views = ctx.arena.grad_views(g)   # fresh views: AccumulateGrad adopts them without a copy
        return (None, None, None) + tuple(v if need else None for v, need in zip(views, ctx.needs))


def _xflag(x: torch.Tensor) -> int:
    return L.X_BF16 if x.dtype == torch.bfloat16 else L.X_F32


class _VAEForward(torch.autograd.Function):
    """``VAEModel.forward`` with a graph (ps_vae/model.py:38-63 under autograd): the forward pass is one library call; the backward pass
    is ``psvae_vae_backward``, which recomputes the activations from the saved input and the same noise draw and back-propagates the
    caller's d loss / d (x_hat, mu, log_sigma) through decoder, reparameterisation and both encoders in the fused kernels."""

    @staticmethod
    def forward(ctx, hot: "HotPath", x: torch.Tensor, eps: Optional[torch.Tensor], *params):
        x_hat, mu, ls, saved = hot._forward_raw(x, eps)
        ctx.hot, ctx.saved = hot, saved
        ctx.needs = [p.requires_grad for p in params]
        return x_hat, mu, ls

    @staticmethod
    def backward(ctx, g_xhat, g_mu, g_ls):
        hot = ctx.hot
        x, eps, seed, off, row0 = ctx.saved
        dev = x.device
        flat = hot.arena.ensure()
        B = x.shape[0]
        gflat = torch.empty(hot.arena.numel, dtype=torch.float32, device=dev)        # a buffer of its own: autograd adopts / accumulates the views
        gs = [None if g is None else g.detach().to(torch.float32).contiguous() for g in (g_xhat, g_mu, g_ls)]
        with _on(dev):
            ws = hot._workspace(dev, B, L.MODE_TRAIN)
            rc = L.lib().psvae_vae_backward(hot._dref, flat.data_ptr(), hot._shadow(), gflat.data_ptr(), x.data_ptr(), _xflag(x), L.ptr(eps), seed, off,
                                            row0, B, hot.precision, L.ptr(gs[0]), L.ptr(gs[1]), L.ptr(gs[2]), ws.data_ptr(), ws.numel(), _stream_ptr(dev))
        L.check(rc, "psvae_vae_backward")
        views = [gflat[o:o + p.numel()].view(p.shape) for p, o in hot.vae_entries()]
        return (None, None, None) + tuple(v if need else None for v, need in zip(views, ctx.needs))


class HotPath:
    """Everything the drop-in modules ask of the CUDA library, for one (VAE [+ latent classifier]) pair."""

    def __init__(self, vae: nn.Module, classifier: Optional[nn.Module] = None, precision: str = "fp32"):
        self.vae = vae
        self.classifier = classifier
        self.set_precision(precision)
        heads: List[int] = []
        self.head_names: List[Optional[str]] = []
        n_trunk, c_hidden, act, single = 0, 0, "relu", True
        if classifier is not None:
            n_trunk = classifier.num_trunk_linears
            c_hidden = classifier.hidden_dim if n_trunk else 0
            act = classifier.activation
            single = classifier.single_label_mode
            heads = list(classifier.head_classes)
            self.head_names = list(classifier.head_names)
            if classifier.input_dim != vae.latent_dim:
                raise ValueError(f"classifier input_dim={classifier.input_dim} must equal the VAE latent_dim={vae.latent_dim}")
        self.desc = L.make_desc(vae.input_dim, vae.latent_dim, vae.hidden_dim, vae.num_hidden_layers, vae.normalize_decoder,
                                n_trunk, c_hidden, act, heads, single)
        self.arena = ParamArena(self.desc, self._entries())
        self._ws: Dict[torch.device, torch.Tensor] = {}
        self._ws_need: Dict[Tuple[int, int, int, int], int] = {}      # psvae_workspace_bytes by (rows, precision, mode, options epoch)
        self._losses: Dict[torch.device, torch.Tensor] = {}
        self.seed: Optional[int] = None
        self.offset = 0            # Philox offset: one per stochastic call
        self.row0 = 0              # global index of this rank's first row (data parallel: rank * local_batch)
        self.flops_train = int(L.lib().psvae_flops_per_sample(self._dref, 0))
        self.flops_forward = int(L.lib().psvae_flops_per_sample(self._dref, 1))
        self.flops_decode = int(L.lib().psvae_flops_per_sample(self._dref, 2))

    # ---- copies ---------------------------------------------------------------------------------
    def __deepcopy__(self, memo):
        """A copy of the owning module gets a HotPath of its own around the COPIED sub-modules: fresh arena (nn.Parameter copies are
        clones, not views), no shared scratch."""
        new = object.__new__(HotPath)
        memo[id(self)] = new
        # the sub-modules may still be under construction at this point (the module being copied reaches its HotPath through its own
        # attributes): the arena is laid out on first use instead (__getattr__)
        new.__dict__["_pending"] = (copy.deepcopy(self.vae, memo), copy.deepcopy(self.classifier, memo), self.precision_name, self.seed, self.offset, self.row0)
        return new

    def __getattr__(self, name):          # reached only when normal lookup fails: a deep copy that has not been laid out yet
        pend = self.__dict__.get("_pending")
        if pend is None or name.startswith("__"):
            raise AttributeError(name)
        del self.__dict__["_pending"]
        self.__init__(*pend[:3])
        self.seed, self.offset, self.row0 = pend[3:]
        return getattr(self, name)

    def __getstate__(self):
        st = dict(self.__dict__)
        st.update(_ws={}, _losses={})
        return st

    # ---- plumbing -------------------------------------------------------------------------------
    @property
    def _dref(self):
        """byref of the model description, built per call (a cached ctypes CArgObject would make the owning module un-copyable / un-picklable)."""
        return C.byref(self.desc)

    def set_precision(self, precision: str) -> None:
        key = str(precision).lower()
        if key not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(set(PRECISIONS))}, got {precision!r}")
        self.precision = PRECISIONS[key]
        self.precision_name = "bf16" if self.precision == L.BF16 else "fp32"

    def _entries(self) -> List[Tuple[nn.Parameter, int]]:
        d, v = self.desc, self.vae
        out: List[Tuple[nn.Parameter, int]] = []
        mu_lin, sg_lin, dec_lin = v.linears("encoder_mu"), v.linears("encoder_sigma"), v.linears("decoder")
        for j, (a, b) in enumerate(zip(mu_lin, sg_lin)):
            out += [(a.weight, d.enc_w[j]), (b.weight, d.enc_w[j] + a.weight.numel()), (a.bias, d.enc_b[j]), (b.bias, d.enc_b[j] + a.bias.numel())]
        for j, a in enumerate(dec_lin):
            out += [(a.weight, d.dec_w[j]), (a.bias, d.dec_b[j])]
        c = self.classifier
        if c is not None:
            for t, lin in enumerate(c.trunk_linears()):
                out += [(lin.weight, d.clf_trunk_w[t]), (lin.bias, d.clf_trunk_b[t])]
            for h, lin in enumerate(c.head_linears()):
                out += [(lin.weight, d.clf_head_w[h]), (lin.bias, d.clf_head_b[h])]
        return out

    def parameters(self) -> List[nn.Parameter]:
        return [p for p, _ in self.arena.entries]

    def _device(self) -> torch.device:
        dev = self.arena.device
        if dev.type != "cuda":
            raise RuntimeError(
                f"pseudo_speaker_vae_b200 runs on a B200 only (module is on {dev}); move it with .to('cuda'). There is no CPU fallback.")
        return dev

    def _workspace(self, dev: torch.device, rows: int, mode: int, extra: int = 0) -> torch.Tensor:
        key = (rows, self.precision, mode, L.OPTIONS_EPOCH)
        need = self._ws_need.get(key)
        if need is None:
            need = int(L.lib().psvae_workspace_bytes(self._dref, rows, self.precision, mode))
            if need < 0:
                raise ValueError(L.last_error())
            if len(self._ws_need) > 64:
                self._ws_need.clear()
            self._ws_need[key] = need
        need += extra
        ws = self._ws.get(dev)
        if ws is None or ws.numel() < need:
            self._ws[dev] = ws = torch.empty(need, dtype=torch.uint8, device=dev)
        return ws

    def _rng(self) -> Tuple[int, int]:
        if self.seed is None:
            self.seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
        off = self.offset
        self.offset += 1
        return self.seed, off

    def manual_seed(self, seed: int, offset: int = 0) -> None:
        self.seed, self.offset = int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset)

    def _shadow(self) -> Optional[int]:
        return self.arena.shadow_ptr(self._dref) if self.precision == L.BF16 else None

    @staticmethod
    def _f32(t: torch.Tensor, dev: torch.device, what: str) -> torch.Tensor:
        if t.device != dev:
            raise ValueError(f"{what} is on {t.device}, the model on {dev}")
        return t.detach().to(torch.float32).contiguous()

    def _x_in(self, x: torch.Tensor, dev: torch.device, plain_tail: bool = True) -> torch.Tensor:
        """The input batch as the library takes it: fp32, or -- tensor-core mode with the plain MSE tail -- bf16 as it is (a batch from a
        bf16 embedding store: no cast pass on the device, half the H2D bytes; the bf16 values are the data)."""
        if x.device != dev:
            raise ValueError(f"x is on {x.device}, the model on {dev}")
        if x.dtype == torch.bfloat16 and self.precision == L.BF16 and plain_tail:
            return x.detach().contiguous()
        return x.detach().to(torch.float32).contiguous()

    # ---- VAEModel.forward (ps_vae/model.py:38-63) -------------------------------------------------
    def vae_entries(self) -> List[Tuple[nn.Parameter, int]]:
        """(parameter, arena offset) of the VAE's own parameters (the classifier's follow them in the arena)."""
        return [(p, o) for p, o in self.arena.entries if o < int(self.desc.vae_numel)]

    def forward(self, x: torch.Tensor, eps: Optional[torch.Tensor] = None):
        """(x_hat, mu, log_sigma).  With autograd on and trainable VAE parameters the outputs carry a graph, as the reference's do: a
        caller's own loss on them back-propagates through ``psvae_vae_backward``.  (``training_step`` does not come through here: it
        computes its loss and every gradient in one fused call.)"""
        entries = self.vae_entries()
        if torch.is_grad_enabled() and x.dim() == 2 and x.shape[0] > 0 and any(p.requires_grad for p, _ in entries):
            if x.requires_grad:
                raise NotImplementedError("the gradient with respect to the input x is not computed by the B200 path (model parameters only)")
            return _VAEForward.apply(self, x, eps, *[p for p, _ in entries])
        x_hat, mu, ls, _ = self._forward_raw(x, eps)
        return x_hat, mu, ls

    def _forward_raw(self, x: torch.Tensor, eps: Optional[torch.Tensor] = None):
        dev = self._device()
        flat = self.arena.ensure()
        if x.dim() != 2 or x.shape[1] != self.desc.input_dim:
            raise ValueError(f"x must be [batch, {self.desc.input_dim}], got {tuple(x.shape)}")
        x = self._x_in(x, dev)
        B = x.shape[0]
        D, Lz = self.desc.input_dim, self.desc.latent_dim
        x_hat = torch.empty(B, D, dtype=torch.float32, device=dev)
        mu = torch.empty(B, Lz, dtype=torch.float32, device=dev)
        ls = torch.empty(B, Lz, dtype=torch.float32, device=dev)
        if B == 0:
            return x_hat, mu, ls, None
        if eps is not None:
            eps = self._f32(eps, dev, "eps")
            if tuple(eps.shape) != (B, Lz):
                raise ValueError(f"eps must be [{B}, {Lz}], got {tuple(eps.shape)}")
            seed, off = 0, 0
        else:
            seed, off = self._rng()
        with _on(dev):
            ws = self._workspace(dev, B, L.MODE_FORWARD)
            rc = L.lib().psvae_forward(self._dref, flat.data_ptr(), self._shadow(), x.data_ptr(), _xflag(x), L.ptr(eps), seed, off, self.row0, B,
                                       self.precision, x_hat.data_ptr(), mu.data_ptr(), ls.data_ptr(), ws.data_ptr(), ws.numel(), _stream_ptr(dev))
        L.check(rc, "psvae_forward")
        return x_hat, mu, ls, (x, eps, seed, off, self.row0)      # what the backward pass needs to redo this exact forward

    # ---- VAEModel.decode (model.py:65-69) / unconditional_synthesis (inference.py:22-25) ----------
    def decode(self, z: Optional[torch.Tensor], num_samples: Optional[int] = None, out: Optional[torch.Tensor] = None,
               return_z: bool = False, row0: Optional[int] = None):
        dev = self._device()
        flat = self.arena.ensure()
        D, Lz = self.desc.input_dim, self.desc.latent_dim
        if z is not None:
            if z.dim() != 2 or z.shape[1] != Lz:
                raise ValueError(f"z must be [n, {Lz}], got {tuple(z.shape)}")
            z = self._f32(z, dev, "z")
            N = z.shape[0]
            seed, off = 0, 0
        else:
            N = int(num_samples)
            seed, off = self._rng()
        if out is None:
            out = torch.empty(N, D, dtype=torch.float32, device=dev)
        elif tuple(out.shape) != (N, D) or out.dtype != torch.float32 or not out.is_contiguous() or out.device != dev:
            raise ValueError(f"out must be a contiguous float32 [{N}, {D}] tensor on {dev}")
        z_out = torch.empty(N, Lz, dtype=torch.float32, device=dev) if (return_z and z is None) else None
        if N > 0:
            with _on(dev):
                ws = self._workspace(dev, N, L.MODE_DECODE)
                rc = L.lib().psvae_decode(self._dref, flat.data_ptr(), self._shadow(), L.ptr(z), seed, off, self.row0 if row0 is None else row0, N,
                                          self.precision, out.data_ptr(), L.ptr(z_out), ws.data_ptr(), ws.numel(), _stream_ptr(dev))
            L.check(rc, "psvae_decode")
        if return_z:
            return out, (z if z is not None else z_out)
        return out

    # ---- training_step / validation_step (lightning.py:67-197) + backward -------------------------
    def pack_labels(self, y, rows: int, dev: torch.device) -> Optional[torch.Tensor]:
        """int64 [num_heads][rows]; single-label: the tensor itself; multi-label: {label: tensor} in head order."""
        if self.classifier is None:
            return None
        if isinstance(y, dict):
            if self.classifier.single_label_mode:
                raise ValueError("labels must be a tensor for a single-label classifier")
            cols = [y[name] for name in self.head_names]
            y = torch.stack([c.to(device=dev, dtype=torch.int64).reshape(-1) for c in cols], 0)
        else:
            if not self.classifier.single_label_mode:
                raise ValueError("labels must be a dict {label: tensor} for a multi-label classifier")
            y = y.to(device=dev, dtype=torch.int64).reshape(1, -1)
        if y.shape[1] != rows:
            raise ValueError(f"labels have {y.shape[1]} rows, x has {rows}")
        return y.contiguous()

    def step(self, x: torch.Tensor, y=None, eps: Optional[torch.Tensor] = None, *, kl_weight: float = 1.0, clf_weight: float = 1.0,
             use_cos_loss: bool = False, compute_grads: bool = True, grads: Optional[torch.Tensor] = None, want_outputs: bool = False,
             consistency: Optional[nn.Module] = None, consistency_y: Optional[torch.Tensor] = None, consistency_weight: float = 1.0,
             counters: Optional[torch.Tensor] = None, accumulate: bool = False, grad_scratch: Optional[torch.Tensor] = None,
             grad_scope: str = "all"):
        """One fused forward(+backward), ``psvae_train_fwd_bwd_scoped``.  Returns (losses[16] device tensor, flat grads or None, outputs or
        None).

        ``consistency``: a frozen ``EmbeddingClassifier`` whose ``consistency_weight * CE(consistency(x_hat), consistency_y)``
        joins the loss (lightning.py:100-108, 119-124).  losses slots: _lib.LOSS_*; nothing here synchronises with the host.
        ``counters``: a device ``psvae_step_counters`` block (int64 [_lib.COUNTER_SLOTS]); the Philox offset of the eps draw is then read
        from it on the device, so that a CUDA graph of this call draws fresh noise at every replay.  The host offset still advances as
        usual: it is the mirror the caller keeps the block in step with.
        ``accumulate``: ADD this batch's gradients to what ``grads`` holds (they are computed into ``grad_scratch``, a flat fp32 buffer of
        the arena's size, then added with one fp32 addition per element).
        ``grad_scope``: ``"all"``, or ``"classifier"`` for a frozen VAE (``train_scope()``): the same forward and losses, but only the latent
        classifier's gradients are computed, and only the classifier span of ``grads`` (``classifier_span()``) is written -- or, with
        ``accumulate``, added to; every other element of ``grads`` keeps its value."""
        if grad_scope not in ("all", "classifier"):
            raise ValueError(f"grad_scope must be 'all' or 'classifier', got {grad_scope!r}")
        if grad_scope == "classifier" and self.classifier is None:
            raise ValueError("grad_scope 'classifier' needs a model with a latent classifier")
        clf_scope = compute_grads and grad_scope == "classifier"
        dev = self._device()
        flat = self.arena.ensure()
        D, Lz = self.desc.input_dim, self.desc.latent_dim
        if x.dim() != 2 or x.shape[1] != D:
            raise ValueError(f"x must be [batch, {D}], got {tuple(x.shape)}")
        x = self._x_in(x, dev, plain_tail=not (self.desc.normalize_decoder or use_cos_loss or consistency is not None))
        B = x.shape[0]
        if B == 0:
            raise ValueError("empty batch")
        yy = self.pack_labels(y, B, dev)
        if eps is not None:
            eps = self._f32(eps, dev, "eps")
            if tuple(eps.shape) != (B, Lz):
                raise ValueError(f"eps must be [{B}, {Lz}], got {tuple(eps.shape)}")
            seed, off = 0, 0
        else:
            seed, off = self._rng()
        losses = torch.empty(L.NUM_LOSSES, dtype=torch.float32, device=dev)
        if compute_grads and grads is None:
            grads = self.arena.stage_buffer()
        outs = None
        xh = mu = ls = None
        if want_outputs:
            xh = torch.empty(B, D, dtype=torch.float32, device=dev)
            mu = torch.empty(B, Lz, dtype=torch.float32, device=dev)
            ls = torch.empty(B, Lz, dtype=torch.float32, device=dev)
            outs = (xh, mu, ls)
        mode = L.MODE_TRAIN_CLASSIFIER if clf_scope else L.MODE_TRAIN if compute_grads else L.MODE_FORWARD
        args = (self._dref, flat.data_ptr(), self._shadow(), L.ptr(grads) if compute_grads else None, x.data_ptr(), _xflag(x), L.ptr(yy),
                L.ptr(eps), seed, off, self.row0, B, float(kl_weight), float(clf_weight), int(bool(use_cos_loss)),
                int(bool(compute_grads)), self.precision, L.ptr(xh), L.ptr(mu), L.ptr(ls), losses.data_ptr())
        cons_args = (None, None, None, 0.0)
        if consistency is not None:
            if consistency.input_dim != D:
                raise ValueError(f"consistency classifier input_dim={consistency.input_dim} must equal the VAE input_dim={D}")
            if consistency_y is None or isinstance(consistency_y, dict):
                raise ValueError("the consistency classifier needs single-label targets (a tensor)")
            cy = consistency_y.to(device=dev, dtype=torch.int64).reshape(-1).contiguous()
            if cy.numel() != B:
                raise ValueError(f"labels have {cy.numel()} rows, x has {B}")
            cdesc, cflat = consistency.flat_params(dev)
            extra = int(L.lib().psvae_consistency_workspace_bytes(C.byref(cdesc), B, L.MODE_FORWARD if clf_scope else mode))
            if extra < 0:
                raise ValueError(L.last_error())
            cons_args = (C.byref(cdesc), cflat.data_ptr(), cy.data_ptr(), float(consistency_weight))
        if counters is not None and (counters.device != dev or counters.dtype != torch.int64 or counters.numel() != L.COUNTER_SLOTS):
            raise ValueError(f"counters must be an int64 [{L.COUNTER_SLOTS}] tensor on {dev}")
        acc = bool(accumulate and compute_grads)
        if acc:
            if grads is None or grad_scratch is None or grad_scratch.device != dev or grad_scratch.dtype != torch.float32 \
                    or grad_scratch.numel() < self.arena.numel or grad_scratch.data_ptr() == grads.data_ptr():
                raise ValueError("an accumulating step needs `grads` and a separate fp32 `grad_scratch` of the arena's size on the same device")
        with _on(dev):
            ws = self._workspace(dev, B, mode, extra if consistency is not None else 0)
            rc = L.lib().psvae_train_fwd_bwd_scoped(*args, ws.data_ptr(), ws.numel(), _stream_ptr(dev), *cons_args, L.ptr(counters), int(acc),
                                                    L.ptr(grad_scratch) if acc else None, L.GRAD_CLASSIFIER if clf_scope else L.GRAD_ALL)
        L.check(rc, "psvae_train_fwd_bwd_scoped")
        return losses, (grads if compute_grads else None), outs

    def train_scope(self) -> str:
        """The gradient scope the ``requires_grad`` flags call for: ``"classifier"`` when every VAE parameter is frozen and every classifier
        parameter is trainable (the second stage of a two-stage run, ``freeze_vae``), ``"all"`` for any other mix."""
        if self.classifier is None:
            return "all"
        vae_numel = int(self.desc.vae_numel)
        vae = [p.requires_grad for p, o in self.arena.entries if o < vae_numel]
        clf = [p.requires_grad for p, o in self.arena.entries if o >= vae_numel]
        return "classifier" if not any(vae) and all(clf) else "all"

    def classifier_span(self) -> Tuple[int, int]:
        """[a, b) of the classifier's parameters (and the arena's tail padding) in the flat buffers: what the classifier scope writes."""
        return int(self.desc.vae_numel), int(self.desc.total_numel)

    def loss_with_grad(self, losses: torch.Tensor, gflat: torch.Tensor) -> torch.Tensor:
        """The scalar a LightningModule returns from training_step: ``.backward()`` hands the fused gradients to autograd."""
        params = self.parameters()
        return _FusedLoss.apply(losses[L.LOSS_TOTAL], gflat, self.arena, *params)

    # ---- conditional_synthesis Langevin loop (inference.py:72-103) --------------------------------
    def targets_for(self, classifier_target) -> List[int]:
        c = self.classifier
        if c is None:
            raise ValueError("conditional synthesis needs a model with a latent classifier")
        if c.single_label_mode:
            if isinstance(classifier_target, dict):
                raise ValueError("classifier_target must be an int for a single-label classifier")
            t = int(classifier_target)
            if not 0 <= t < c.head_classes[0]:
                raise IndexError(f"classifier_target {t} is out of range for {c.head_classes[0]} classes")
            return [t]
        assert isinstance(classifier_target, dict), "classifier_target must be a dict for multi-label classifier"
        out = []
        for name, ncls in zip(self.head_names, c.head_classes):
            if name in classifier_target:
                t = int(classifier_target[name])
                if not 0 <= t < ncls:
                    raise IndexError(f"classifier_target[{name!r}]={t} is out of range for {ncls} classes")
                out.append(t)
            else:
                out.append(-1)
        unknown = [k for k in classifier_target if k not in self.head_names]
        if unknown:
            raise KeyError(unknown[0])
        return out

    def row_targets_for(self, classifier_target, num_samples: int, device, check: bool = False) -> Optional[torch.Tensor]:
        """The device int32 ``[n_heads][N]`` targets of a per-row ``classifier_target``, or None for a shared one (an int, a 0-d tensor, a
        dict of ints).  Per row: a 1-D integer tensor / array of length N (single-label), or a dict whose values are ints (broadcast) or
        length-N integer tensors (multi-label); a label the dict leaves out, and -1 inside a tensor, leave that head out for the row.
        ``check`` validates the values on the host (one synchronisation) and raises IndexError / ValueError as ``targets_for`` does;
        without it a bad row comes out of the kernel as NaN."""
        def per_row(v):
            return isinstance(v, (torch.Tensor, np.ndarray)) and v.ndim >= 1

        def vec(v, what):
            t = v if isinstance(v, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(v))
            if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
                raise TypeError(f"{what} must be an integer tensor, got {t.dtype}")
            if t.dim() != 1 or t.shape[0] != N:
                raise ValueError(f"{what} must be 1-D with {N} rows, got shape {tuple(t.shape)}")
            # clamp before the int32 cast so that no out-of-range value wraps into a valid class
            return t.to(device=device, dtype=torch.int64, non_blocking=True).clamp(-2, 127).to(torch.int32)

        c = self.classifier
        if c is None:
            raise ValueError("conditional synthesis needs a model with a latent classifier")
        N = int(num_samples)
        if isinstance(classifier_target, dict):
            if not any(per_row(v) for v in classifier_target.values()):
                return None
            if c.single_label_mode:
                raise ValueError("classifier_target must be an int or a 1-D tensor for a single-label classifier")
            unknown = [k for k in classifier_target if k not in self.head_names]
            if unknown:
                raise KeyError(unknown[0])
            out = torch.full((len(c.head_classes), N), -1, dtype=torch.int32, device=device)
            for h, (name, ncls) in enumerate(zip(self.head_names, c.head_classes)):
                if name not in classifier_target:
                    continue
                v = classifier_target[name]
                if per_row(v):
                    out[h] = vec(v, f"classifier_target[{name!r}]")
                else:
                    t = int(v)
                    if not 0 <= t < ncls:
                        raise IndexError(f"classifier_target[{name!r}]={t} is out of range for {ncls} classes")
                    out[h] = t
        elif per_row(classifier_target):
            if not c.single_label_mode:
                raise ValueError("classifier_target must be a dict for a multi-label classifier")
            out = vec(classifier_target, "classifier_target").reshape(1, N)
        else:
            return None
        if check and N > 0:
            host = out.cpu().to(torch.int64)
            for h, (name, ncls) in enumerate(zip(self.head_names, c.head_classes)):
                bad = ((host[h] < -1) | (host[h] >= ncls)).nonzero()
                if bad.numel():
                    i = int(bad[0])
                    what = "classifier_target" if c.single_label_mode else f"classifier_target[{name!r}]"
                    raise IndexError(f"{what} of row {i} is {int(host[h, i])}: out of range for {ncls} classes")
            none = (host < 0).all(dim=0).nonzero()
            if none.numel():
                raise ValueError(f"row {int(none[0])} of classifier_target names no head")
        return out

    def target_mix_for(self, target_mix) -> Tuple[List[List[int]], List[int]]:
        """The entries (targets per head, -1 = left out) and uint32 thresholds of ``target_mix = [(target, weight), ...]``: each target is
        what the shared form accepts, zero-weight entries are dropped (utils.mix_thresholds)."""
        from .utils import mix_thresholds

        pairs = list(target_mix)
        if not pairs:
            raise ValueError("target_mix is empty")
        for p in pairs:
            if not isinstance(p, (tuple, list)) or len(p) != 2:
                raise ValueError(f"target_mix entry {p!r} is not a (target, weight) pair")
        kept, thr = mix_thresholds([w for _, w in pairs], L.MAX_TARGET_MIX)
        return [self.targets_for(pairs[i][0]) for i in kept], thr

    def _targets_out(self, t: torch.Tensor):
        """int32 [n_heads][N] kernel targets -> int64 [N] (single-label) or {label: int64 [N]}."""
        if self.classifier.single_label_mode:
            return t[0].to(torch.int64)
        return {name: t[h].to(torch.int64) for h, name in enumerate(self.head_names)}

    def langevin(self, num_samples: int, classifier_target, step_size: float = 0.01, num_steps: int = 100, noise_weight: float = 1.0,
                 z0: Optional[torch.Tensor] = None, noise: Optional[torch.Tensor] = None, return_history: bool = False, return_stats: bool = False,
                 row0: Optional[int] = None, prior_weight: float = 1.0, threshold: float = 0.0, return_stop: bool = False, *,
                 target_mix=None, check_targets: bool = False):
        """The Langevin loop of inference.py:72-103 in one launch.  ``prior_weight`` / ``threshold`` / ``return_stop`` cover the analysis variant
        (analysis/sample_gender_transformation.py:61-99): the log p(z) term scaled by ``prior_weight``, a sample frozen after the update of the
        first step whose p(y|z) exceeded ``threshold`` (0 = never); with ``return_stop`` the third result is ``(stats, stop_step, last_prob)``.

        ``classifier_target`` is shared (int, dict of ints) or per row (see ``row_targets_for``; ``check_targets`` validates it on the host).
        ``target_mix = [(target, weight), ...]`` (with ``classifier_target=None``) draws each row's target in the kernel from the global row
        index; the drawn targets come back as a fourth result (``_targets_out`` form) and the call uses ``num_steps + 2`` Philox offsets."""
        dev = self._device()
        flat = self.arena.ensure()
        Lz = self.desc.latent_dim
        N = int(num_samples)
        rows_t = mix = None
        if target_mix is not None:
            if classifier_target is not None:
                raise ValueError("give either classifier_target or target_mix, not both")
            if self.classifier is None:
                raise ValueError("conditional synthesis needs a model with a latent classifier")
            mix = self.target_mix_for(target_mix)
        else:
            if classifier_target is None:
                raise ValueError("conditional synthesis needs a classifier_target or a target_mix")
            rows_t = self.row_targets_for(classifier_target, N, dev, check_targets)
        if mix is None and rows_t is None:
            targets = self.targets_for(classifier_target)
            tarr = (C.c_int32 * L.MAX_CLF_HEADS)(*(targets + [-1] * (L.MAX_CLF_HEADS - len(targets))))
        if z0 is not None:
            z = self._f32(z0, dev, "z0").clone()
            if tuple(z.shape) != (N, Lz):
                raise ValueError(f"z0 must be [{N}, {Lz}]")
            init = 0
        else:
            z = torch.empty(N, Lz, dtype=torch.float32, device=dev)
            init = 1
        if noise is not None:
            noise = self._f32(noise, dev, "noise")
            if tuple(noise.shape) != (num_steps, N, Lz):
                raise ValueError(f"noise must be [{num_steps}, {N}, {Lz}]")
        if self.seed is None:
            self.seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
        off0 = self.offset
        self.offset += num_steps + (2 if mix is not None else 1)
        hist = torch.empty(num_steps, N, Lz, dtype=torch.float32, device=dev) if return_history else None
        stats = torch.empty(num_steps, 2, dtype=torch.float32, device=dev) if return_stats else None
        stop = torch.full((N,), int(num_steps), dtype=torch.int32, device=dev) if return_stop else None
        prob = torch.zeros(N, dtype=torch.float32, device=dev) if return_stop else None
        tout = torch.empty(len(self.classifier.head_classes), N, dtype=torch.int32, device=dev) if mix is not None else None
        r0 = self.row0 if row0 is None else row0
        if N > 0 and mix is None and rows_t is None:
            with _on(dev):
                rc = L.lib().psvae_langevin(self._dref, flat.data_ptr(), z.data_ptr(), N, tarr, float(step_size), int(num_steps), float(noise_weight),
                                            self.seed, off0, r0, init, L.ptr(noise), L.ptr(hist), L.ptr(stats),
                                            float(prior_weight), float(threshold), L.ptr(stop), L.ptr(prob), _stream_ptr(dev))
            L.check(rc, "psvae_langevin")
        elif N > 0:
            n_mix, marr, tharr = 0, None, None
            if mix is not None:
                entries, thr = mix
                n_mix = len(entries)
                marr = (C.c_int32 * (n_mix * L.MAX_CLF_HEADS))(*[t for e in entries for t in e + [-1] * (L.MAX_CLF_HEADS - len(e))])
                tharr = (C.c_uint32 * max(1, len(thr)))(*thr)
            with _on(dev):
                rc = L.lib().psvae_langevin_rows(self._dref, flat.data_ptr(), z.data_ptr(), N, L.ptr(rows_t), n_mix, marr, tharr, L.ptr(tout),
                                                 float(step_size), int(num_steps), float(noise_weight), self.seed, off0, r0, init, L.ptr(noise),
                                                 L.ptr(hist), L.ptr(stats), float(prior_weight), float(threshold), L.ptr(stop), L.ptr(prob),
                                                 _stream_ptr(dev))
            L.check(rc, "psvae_langevin_rows")
        if stats is not None and N > 0:
            stats = stats / N
        res = (z, hist, (stats, stop, prob) if return_stop else stats)
        if mix is not None:
            return res + (self._targets_out(tout),)
        return res
