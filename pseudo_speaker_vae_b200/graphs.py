"""``GraphedTrainStep`` -- the data-parallel train step (fused forward + backward -> gradient all-reduce -> fused Adam) replayed as ONE
CUDA graph.

At small batches (the reference trains at about 2,048 rows; strong scaling over 8 GPUs lands at 8,192 per rank) the fixed cost of a step
is a large share of it: the Python of ``HotPath.step``, the library's launches, the all-reduce and the optimiser's loop over spans are
enqueued by the host every step.  A graph enqueues them once.  The three values that change every step and used to be frozen into kernel
arguments -- the Philox offset of the eps draw, Adam's step count and the learning rate -- live in device memory here
(``psvae_step_counters`` + one fp64 lr per parameter group), so a replay computes exactly what the eager ``DataParallelTrainer.train_step``
computes (bit for bit in the deterministic summation mode).

Opt-in, because the call contract changes: the batch is copied into static input buffers, and the returned loss tensor is the graph's
static output -- the next call overwrites it.

    trainer = DataParallelTrainer(module)
    step = GraphedTrainStep(trainer, rows=2048)
    for x, y in loader:
        losses = step(x, y)        # call 1 eager (warm-up), call 2 captures + replays, later calls replay; another row count runs eagerly
        sched.step()               # lr changes reach the graph through the device lr array

The host keeps its usual view of the run -- ``hot_path.offset``, ``optimizer.state[p]['step']``, the arena epoch and the bf16 shadow
mark -- by counting replays (no read-back), so eager steps, ``state_dict()`` and checkpoints in between see the right values; whenever
those host values differ from what the device block holds (a scheduler step, ``load_state_dict``, an eager step, ``manual_seed``) the
host values are written to the block before the next replay.

With the trainer's ``accumulate_grad_batches = k`` each call is one micro-batch, and up to three graphs are captured, each on first use:
the first micro-batch of a window (writes the gradient buffer), a middle one (adds to it) and the last one (adds, then all-reduce, norm
clipping, Adam).  With k = 1 there is one graph, as without the option.  Every replay advances the Philox offset; only the last one
advances the Adam step.  ``flush=True`` ends the window early, as it does for ``DataParallelTrainer.train_step``.
"""
from __future__ import annotations

import warnings
from typing import Dict, Optional, Tuple

import torch

from . import _lib as L
from .engine import _on, _stream_ptr
from .optim import FusedAdam
from .parallel import DataParallelTrainer


class GraphedTrainStep:
    def __init__(self, trainer: DataParallelTrainer, rows: int, x_dtype: Optional[torch.dtype] = None):
        """``x_dtype``: element type of the static input buffer (None: the dtype of the batch the graph is captured with).  A batch of
        another dtype is refused rather than converted, so that a replay computes what the eager step computes on the same batch."""
        self.trainer = trainer
        self.hot = trainer.hot
        self.optimizer = trainer.optimizer
        self.rows = int(rows)
        self.x_dtype = x_dtype
        self.device = self.hot._device()           # no CPU fallback: a module off the GPU raises here
        n_groups = len(self.optimizer.param_groups)
        self.counters = torch.zeros(n_groups, L.COUNTER_SLOTS, dtype=torch.int64, device=self.device)
        self.lrs = torch.zeros(n_groups, dtype=torch.float64, device=self.device)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.losses: Optional[torch.Tensor] = None  # the graph's static output
        self._graphs: Dict[Tuple[bool, bool], Tuple[torch.cuda.CUDAGraph, torch.Tensor]] = {}   # (accumulate, step) -> (graph, losses)
        self.replays = 0
        self.pdl: Optional[int] = None             # 1: captured with programmatic dependent launch; 0: captured without it
        self.capture_error: Optional[str] = None   # why a first capture attempt failed (kept when a fallback capture succeeded)
        self.allreduce_kind: Optional[str] = None  # the all-reduce the graph contains ("none" on one rank)
        self._warm = False
        self._key = None
        self._mirror = None                        # the host values the device block holds
        self._static: Dict[str, object] = {}

    # ---- host <-> device state ------------------------------------------------------------------
    def _host_values(self) -> Tuple:
        opt = self.optimizer
        steps = tuple(int(opt.state[g["params"][0]]["step"]) if "step" in opt.state[g["params"][0]] else 0 for g in opt.param_groups)
        return (int(self.hot.offset), steps, tuple(float(g["lr"]) for g in opt.param_groups))

    def _sync_device(self) -> None:
        vals = self._host_values()
        if vals == self._mirror:
            return
        off, steps, lrs = vals
        c = torch.zeros(len(steps), L.COUNTER_SLOTS, dtype=torch.int64)
        c[:, L.COUNTER_RNG_OFFSET] = off
        c[:, L.COUNTER_ADAM_STEP] = torch.tensor(steps, dtype=torch.int64)
        self.counters.copy_(c)
        self.lrs.copy_(torch.tensor(lrs, dtype=torch.float64))
        self._mirror = vals

    def _advance_mirrors(self, step: bool = True) -> None:
        """What one replay did, on the host: the eager step's _rng() and (``step``) FusedAdam.step() bookkeeping."""
        opt, arena = self.optimizer, self.hot.arena
        self.hot.offset += 1
        if step:
            for g in opt.param_groups:
                opt.state[g["params"][0]]["step"] += 1       # one tensor shared by the group's parameters (FusedAdam._bind_state)
            arena.epoch += 1
            if arena.shadow is not None:
                arena.mark_shadow_current()
        self.trainer._end_micro_batch(step)
        self.replays += 1
        self._mirror = self._host_values()

    def _capture_key(self) -> Tuple:
        """Everything a replay takes as it was at capture: a change of any of it means a new capture."""
        tr, hot, opt = self.trainer, self.hot, self.optimizer
        m = tr.module
        cons = getattr(m, "consistency_classifier", None)
        cflat = cons.flat_params(self.device)[1].data_ptr() if cons is not None else None
        groups = tuple((tuple(g["betas"]), g["eps"], g["weight_decay"], g["amsgrad"], g["maximize"], tuple(id(p) for p in g["params"]))
                       for g in opt.param_groups)
        bufs = (hot.arena.flat.data_ptr(), L.ptr(hot.arena.shadow), opt._m.data_ptr(), opt._v.data_ptr(), L.ptr(opt._vmax),
                tr._views_of.data_ptr() if tr._views_of is not None else None, cflat)
        knobs = (tr.accumulate_grad_batches, tr.gradient_clip_val, tr.gradient_clip_algorithm, opt.clip_mode, opt.clip_value, L.ptr(opt.clip_coef),
                 L.ptr(tr._acc_scratch), L.ptr(tr._norm_scratch))
        trained = tuple(p.requires_grad for p in hot.parameters())      # the gradient scope and the Adam spans follow from it
        return (hot.seed, hot.row0, hot.precision, m.kl_loss_weight, m.classifier_loss_weight, m.use_cos_loss, m.consitency_loss_weight,
                id(cons), L.OPTIONS_EPOCH, opt.grad_scale, groups, bufs, knobs, trained)

    # ---- capture --------------------------------------------------------------------------------
    def _check_supported(self) -> None:
        opt, tr = self.optimizer, self.trainer
        if not isinstance(opt, FusedAdam):
            raise NotImplementedError(f"a graphed train step needs FusedAdam, got {type(opt).__name__}")
        # a frozen VAE (classifier scope) is the one partial freeze a graph takes: Adam rewrites only the classifier, whose slice of the bf16
        # copy no kernel reads, and the VAE's slice stays what the refresh before capture made it
        frozen_vae = self.hot.train_scope() == "classifier" and \
            {id(p) for g in opt.param_groups for p in g["params"] if p.grad is not None} == {id(p) for p in self.hot.parameters() if p.requires_grad}
        if not opt.covers_arena() and not frozen_vae:
            raise NotImplementedError("a graphed train step needs every arena parameter trained (no frozen parameters): the bf16 operand "
                                      "copy must be rewritten by Adam, not refreshed inside the graph")
        if tr._views_of is None or self.hot.arena.flat_grad() is None:
            raise NotImplementedError("a graphed train step reads the gradients from the trainer's flat gradient buffer")

    def _body(self, kind: Optional[str], phase: Tuple[bool, bool] = (False, True)) -> torch.Tensor:
        st, tr = self._static, self.trainer
        accumulate, step = phase
        losses, gflat = tr._fwd_bwd(st["x"], st["y"], None, counters=self.counters[0], accumulate=accumulate)
        if step:
            tr._all_reduce(gflat, kind)
            tr._clip_norm(gflat)
            self.optimizer._update(self.counters, self.lrs)
        lib, stream = L.lib(), _stream_ptr(self.device)
        with _on(self.device):
            for gi in range(self.counters.shape[0]):
                L.check(lib.psvae_step_counters_advance_by(self.counters[gi].data_ptr(), 1, int(step), stream), "psvae_step_counters_advance_by")
        return losses

    def _try_capture(self, kind: Optional[str], pdl: int, phase: Tuple[bool, bool] = (False, True)) -> Tuple[Optional[torch.cuda.CUDAGraph], Optional[torch.Tensor], Optional[BaseException]]:
        off0 = self.hot.offset
        pdl0 = L.get_option("pdl")
        g = torch.cuda.CUDAGraph()
        try:
            if pdl != pdl0:
                L.set_option("pdl", pdl)
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                losses = self._body(kind, phase)
            return g, losses, None
        except Exception as e:  # noqa: BLE001 -- reported by the caller, which may retry with another configuration
            return None, None, e
        finally:
            self.hot.offset = off0        # capture does not execute: the _rng() bump of the captured call is not a step
            if pdl != pdl0:
                L.set_option("pdl", pdl0)

    @staticmethod
    def _label_sig(y):
        if y is None:
            return None
        if isinstance(y, dict):
            return tuple(sorted((k, tuple(v.shape)) for k, v in y.items()))
        return tuple(y.shape)

    def _capture(self, x: torch.Tensor, y, phase: Tuple[bool, bool] = (False, True)) -> None:
        """Capture the graph of one window phase (accumulate, step).  A new static input layout drops the graphs of the other phases."""
        self._check_supported()
        tr, dev, hot = self.trainer, self.device, self.hot
        tr._knob_buffers(dev)
        self.optimizer._moments()          # a window's first graphs may be captured before any Adam step has allocated the moments
        if not self._graphs or self._capture_key() != self._key or self._label_sig(y) != self._static.get("ysig") \
                or x.shape[1] != self._static["x"].shape[1]:
            self._graphs = {}
            self._static = {"x": torch.empty(self.rows, x.shape[1], dtype=self.x_dtype or x.dtype, device=dev), "ysig": self._label_sig(y)}
            if isinstance(y, dict):
                self._static["y"] = {k: torch.empty(v.shape, dtype=torch.int64, device=dev) for k, v in y.items()}
            else:
                self._static["y"] = None if y is None else torch.empty(tuple(y.shape), dtype=torch.int64, device=dev)
        self._copy_in(x, y)
        hot._shadow()                      # the graph contains no shadow refresh: the copy must be current before capture
        self.graph = self.losses = None
        torch.cuda.synchronize(dev)
        # the attempts, in order: the all-reduce the trainer picked, NCCL if that was a symmetric-memory kind, then the same without
        # programmatic-launch attributes (a driver that refuses them under capture)
        want = tr.symm.kind if tr.symm is not None else None
        if hot.train_scope() == "classifier":          # the classifier's span goes through NCCL (DataParallelTrainer._all_reduce)
            want = "nccl" if tr.world_size > 1 and not tr.local_only else None
        kinds = [want, "nccl"] if want not in (None, "nccl") else [want]
        pdl0 = L.get_option("pdl")
        attempts = [(k, pdl0) for k in kinds] + ([(k, 0) for k in kinds] if pdl0 else [])
        first_err = err = None
        for kind, pdl in attempts:
            g, losses, err = self._try_capture(kind, pdl, phase)
            if tr.world_size > 1 and not tr.local_only:
                # every rank must replay the same collective
                ok = torch.tensor([0.0 if err is not None else 1.0], device=dev)
                torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN, group=tr.group)
                if float(ok) == 0.0 and err is None:
                    err = RuntimeError("the capture failed on another rank")
            if err is None:
                self.graph, self.losses, self.pdl = g, losses, pdl
                self.allreduce_kind = kind or tr.allreduce_kind
                break
            first_err = first_err or err
        if err is not None:
            raise RuntimeError(f"capturing the train step failed: {first_err!r}; last attempt: {err!r}") from err
        if first_err is not None:
            self.capture_error = repr(first_err)
            warnings.warn(f"GraphedTrainStep: the first capture attempt failed ({first_err!r}); captured with all-reduce "
                          f"{self.allreduce_kind!r}, pdl={self.pdl}", RuntimeWarning)
        self._graphs[phase] = (self.graph, self.losses)
        # buffers the graph writes that HotPath may replace later (a larger eager batch, a forward or decode grows the cached workspace):
        # holding them keeps the captured pointers valid; the eager path then works in the new buffer
        self._static.setdefault("ws", []).append(hot._ws.get(dev))
        cons = getattr(tr.module, "consistency_classifier", None)
        self._static["cons_flat"] = cons.flat_params(dev)[1] if cons is not None else None
        self._key = self._capture_key()

    def _copy_in(self, x: torch.Tensor, y) -> None:
        st = self._static
        st["x"].copy_(x)
        if isinstance(y, dict):
            for k, v in y.items():
                st["y"][k].copy_(v)
        elif y is not None:
            st["y"].copy_(y)

    # ---- the step -------------------------------------------------------------------------------
    def __call__(self, x: torch.Tensor, y=None, *, flush: bool = False) -> torch.Tensor:
        """One micro-batch (one optimiser step without accumulation) on this rank's shard; returns the device tensor of local loss
        scalars (for a replay: the graph's static output, overwritten by the next call).  ``flush``: see DataParallelTrainer.train_step."""
        if x.dim() != 2 or x.shape[0] != self.rows:
            return self.trainer.train_step(x, y, flush=flush)
        static_x = self._static.get("x")
        want = self.x_dtype or (static_x.dtype if static_x is not None else x.dtype)
        if x.dtype != want:
            raise ValueError(f"the graphed step takes {want} batches, got {x.dtype}: a conversion into the static input buffer would change "
                             "what the step computes (x_dtype)")
        if not self._warm:
            self._warm = True
            return self.trainer.train_step(x, y, flush=flush)
        phase = self.trainer._window_phase(flush)
        if self.trainer._views_of is not None:
            self.trainer._bind_grads(self.trainer._views_of)      # the trained set may have changed since the last call (unfreezing)
        if (phase not in self._graphs or self._capture_key() != self._key or self._label_sig(y) != self._static["ysig"]
                or x.shape[1] != static_x.shape[1]):
            self._capture(x, y, phase)
        else:
            self._copy_in(x, y)
            self.hot._shadow()             # refreshed outside the graph if something rewrote the parameters out of band
        self.graph, self.losses = self._graphs[phase]
        self._sync_device()
        self.graph.replay()
        self._advance_mirrors(phase[1])
        return self.losses
