"""Data-parallel training of the fused step: one process per GPU, replicated parameters, batch rows sharded
across ranks, ONE bucketed all-reduce of the flat gradient buffer per step (NCCL over NVLink on the GPU box,
gloo in the CPU tests).  This is what ``Trainer(strategy=DDPStrategy(...))`` does for the reference
(ps_vae/training.py:78; SURVEY 2.3 C1-C4), minus its per-parameter bookkeeping:

  C1  gradient all-reduce   -> ``all_reduce_flat``: SUM over ranks of the arena's flat gradient buffer in
                               ``bucket_bytes`` slices (25 MiB like DDP: 5.13 MB of gradients = one bucket),
                               averaging folded into Adam's ``grad_scale = 1/world``;
  C2  per-metric scalar all-reduces (``sync_dist=True``, 3-7 per step) -> the 16 loss slots ride in ONE small
                               all-reduce (``reduce_losses``), only when somebody asks for them;
  C3  initial parameter broadcast -> ``broadcast_parameters`` (one broadcast of the flat buffer);
  C4  DistributedSampler    -> ``shard_batch``: rank r owns rows [r*B/W, (r+1)*B/W) and tells the kernels its
                               global row offset, so the Philox eps stream does not depend on the world size.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib as L

DEFAULT_BUCKET_BYTES = 25 * 1024 * 1024


def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_batch(global_batch: int, rank: int, world_size: int) -> Tuple[int, int]:
    """(row0, rows) of this rank's contiguous shard; the batch must split evenly (DDP semantics need equal shards
    for the mean of means to equal the global mean)."""
    if global_batch % world_size:
        raise ValueError(f"global batch {global_batch} does not split evenly over {world_size} ranks")
    rows = global_batch // world_size
    return rank * rows, rows


def bucket_slices(numel: int, bucket_bytes: int = DEFAULT_BUCKET_BYTES, elem_bytes: int = 4):
    per = max(1, bucket_bytes // elem_bytes)
    return [(a, min(numel, a + per)) for a in range(0, numel, per)]


def all_reduce_flat(flat: torch.Tensor, bucket_bytes: int = DEFAULT_BUCKET_BYTES, group=None, async_op: bool = False):
    """SUM all-reduce of a flat buffer in buckets.  Returns the work handles when ``async_op``."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return []
    works = []
    for a, b in bucket_slices(flat.numel(), bucket_bytes, flat.element_size()):
        w = dist.all_reduce(flat[a:b], op=dist.ReduceOp.SUM, group=group, async_op=async_op)
        if async_op:
            works.append(w)
    return works


def broadcast_parameters(flat: torch.Tensor, src: int = 0, group=None) -> None:
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.broadcast(flat, src=src, group=group)


def reduce_losses(losses: torch.Tensor, group=None) -> torch.Tensor:
    """Mean over ranks of the packed loss scalars (equal shards): one 64-byte all-reduce instead of 3-7."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        out = losses.clone()
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
        return out / dist.get_world_size(group)
    return losses


class SymmetricAllReduce:
    """The flat gradient buffer in torch symmetric memory (P2P-mapped on every rank of the node) and its all-reduce through
    ``torch.ops.symm_mem.two_shot_all_reduce_`` (reduce-scatter + all-gather over NVLink peer loads/stores) or ``multimem_all_reduce_``
    (NVLS: the reduction happens inside the NVSwitch).  For the 5 MB gradient these are latency-bound like NCCL's ring, but with one
    kernel and no proxy thread.  ``pick()`` TIMES the candidates on the running ranks (20 calls each) and keeps the fastest -- NCCL if it
    wins or if anything about symmetric memory is unavailable on this node."""

    def __init__(self, numel: int, device: torch.device, group=None):
        import torch.distributed._symmetric_memory as symm

        self.group = group if group is not None else dist.group.WORLD
        self.gname = self.group.group_name
        self.buf = symm.empty(numel, dtype=torch.float32, device=device)
        symm.rendezvous(self.buf, self.gname)
        self.buf.zero_()
        self.kind = "nccl"
        self.timings = {}

    def _call(self, kind: str) -> None:
        if kind == "two_shot":
            torch.ops.symm_mem.two_shot_all_reduce_(self.buf, "sum", self.gname)
        elif kind == "multimem":
            torch.ops.symm_mem.multimem_all_reduce_(self.buf, "sum", self.gname)
        else:
            dist.all_reduce(self.buf, op=dist.ReduceOp.SUM, group=self.group)

    def pick(self, iters: int = 20) -> str:
        dev = self.buf.device
        best = None
        for kind in ("nccl", "two_shot", "multimem"):
            ok = torch.ones(1, device=dev)
            try:
                for _ in range(3):
                    self._call(kind)
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                dist.barrier(group=self.group)
                e0.record()
                for _ in range(iters):
                    self._call(kind)
                e1.record()
                torch.cuda.synchronize(dev)
                t = torch.tensor([e0.elapsed_time(e1) / iters * 1e3], device=dev)
            except Exception:  # noqa: BLE001 -- this kind is not available here
                ok.zero_()
                t = torch.tensor([float("inf")], device=dev)
            # every rank must take the same decision: a kind counts only if it worked everywhere; its time is the slowest rank's
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
            us = float(t) if float(ok) > 0 else float("inf")
            self.timings[kind] = us
            if best is None or us < 0.95 * self.timings[best]:        # a challenger must be 5 % faster than the incumbent (NCCL first)
                best = kind
        self.kind = best
        self.buf.zero_()
        return best

    def all_reduce(self) -> None:
        self._call(self.kind)


class DataParallelTrainer:
    """The per-batch body of the reference's fit loop (SURVEY 3.1) as three device-side calls:
    fused fwd+bwd  ->  bucketed all-reduce  ->  fused Adam.  Nothing in ``train_step`` synchronises with the host.

    Two ``Trainer`` options of the reference change what one optimiser step computes; they take Lightning's names, so the keys of
    ``config["trainer"]`` can be passed straight through:

    * ``accumulate_grad_batches = k``: each ``train_step`` is one micro-batch.  The first of a window writes the gradient buffer, the
      others add to it; the k-th call (or one with ``flush=True``, Lightning's last batch of an epoch) runs the all-reduce, the clipping
      and Adam, with ``grad_scale = 1 / (k * world)`` -- Lightning's fixed ``loss / k``, also for a flushed partial window.  Every call
      draws its own eps (one Philox offset), as every ``training_step`` does.
    * ``gradient_clip_val`` / ``gradient_clip_algorithm``: ``"norm"`` is ``clip_grad_norm_(params, val)`` on the averaged gradient (the
      global L2 norm is computed on the device, ``psvae_grad_norm``, and the coefficient is applied inside the Adam pass); ``"value"`` is
      ``clip_grad_value_``.  None or 0 turns clipping off.  ``grad_norm`` holds the pre-clip total norm of the last optimiser step as a
      device fp32 scalar (norm clipping only; nothing reads it back).

    Unlike Lightning, ``p.grad`` keeps the unclipped, all-reduced SUM of the window's micro-batch gradients: the averaging (``1 / (k *
    world)``) and the clipping are applied inside the Adam pass, not to the ``.grad`` tensors."""

    def __init__(self, module, optimizer=None, bucket_bytes: int = DEFAULT_BUCKET_BYTES, group=None, local_only: bool = False, *,
                 accumulate_grad_batches: int = 1, gradient_clip_val: Optional[float] = None, gradient_clip_algorithm: Optional[str] = "norm"):
        """``local_only``: a trainer that never talks to the other ranks even inside an initialised process group (the single-process
        twin ``verify_data_parallel_step`` compares the data-parallel run with)."""
        if isinstance(accumulate_grad_batches, bool) or not isinstance(accumulate_grad_batches, int) or accumulate_grad_batches < 1:
            raise ValueError(f"accumulate_grad_batches must be an int >= 1, got {accumulate_grad_batches!r}")
        algo = "norm" if gradient_clip_algorithm is None else gradient_clip_algorithm
        if algo not in ("norm", "value"):
            raise ValueError(f"gradient_clip_algorithm must be 'norm' or 'value', got {gradient_clip_algorithm!r}")
        clip = 0.0 if gradient_clip_val is None else float(gradient_clip_val)
        if not clip >= 0.0:
            raise ValueError(f"gradient_clip_val must be >= 0 (None or 0 turns clipping off), got {gradient_clip_val!r}")
        self.accumulate_grad_batches = accumulate_grad_batches
        self.gradient_clip_val = clip if clip > 0.0 else None
        self.gradient_clip_algorithm = algo
        self.grad_norm: Optional[torch.Tensor] = None     # device fp32 scalar: pre-clip total norm of the last optimiser step
        self._clip_coef: Optional[torch.Tensor] = None
        self._norm_scratch: Optional[torch.Tensor] = None
        self._acc_scratch: Optional[torch.Tensor] = None
        self._micro = 0                                   # micro-batches of the current accumulation window already run
        self.module = module
        self.hot = module.hot_path
        self.group = group
        self.local_only = bool(local_only)
        self.rank, self.world_size = (0, 1) if self.local_only else world()
        self.bucket_bytes = bucket_bytes
        if optimizer is None:
            optimizer = module.configure_optimizers()["optimizer"]
        self.optimizer = optimizer
        self.optimizer.grad_scale = 1.0 / (self.accumulate_grad_batches * self.world_size)
        if self.gradient_clip_val is not None:
            self.optimizer.clip_mode = self.gradient_clip_algorithm
            self.optimizer.clip_value = self.gradient_clip_val
        if not self.local_only:
            broadcast_parameters(self.hot.arena.ensure(), 0, group)
        self.hot.arena.epoch += 1          # the bf16 operand copy must follow the broadcast values
        self._views = None
        self._views_of = None
        self._views_trained = None
        # N > 1: the gradient buffer lives in symmetric memory when one of its all-reduce kernels beats NCCL on these ranks
        # (PSVAE_ALLREDUCE = auto | nccl | two_shot | multimem)
        self.symm: Optional[SymmetricAllReduce] = None
        self.allreduce_kind = "nccl" if self.world_size > 1 else "none"
        want = os.environ.get("PSVAE_ALLREDUCE", "auto")
        if self.world_size > 1 and not self.local_only and want != "nccl" and self.hot.arena.flat.is_cuda:
            sy = None
            ok = torch.ones(1, device=self.hot.arena.flat.device)
            try:
                sy = SymmetricAllReduce(self.hot.arena.numel, self.hot.arena.flat.device, group)
            except Exception:  # noqa: BLE001 -- no symmetric memory on this node / build
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if float(ok) > 0:
                kind = sy.pick() if want == "auto" else want
                sy.kind = kind
                if kind != "nccl":
                    self.symm = sy
                    self.allreduce_kind = kind
                    self.hot.arena._gbuf.append(sy.buf)        # the arena must know the buffer the .grad views live in (FusedAdam.flat_grad)
                self.allreduce_timings = dict(sy.timings)

    def set_shard(self, global_batch: int) -> Tuple[int, int]:
        row0, rows = shard_batch(global_batch, self.rank, self.world_size)
        self.hot.row0 = row0
        return row0, rows

    def train_step(self, x_local: torch.Tensor, y_local=None, eps_local: Optional[torch.Tensor] = None, *, flush: bool = False) -> torch.Tensor:
        """One micro-batch on this rank's shard (with ``accumulate_grad_batches = 1``: one optimiser step).  Returns the device tensor of
        this micro-batch's local loss scalars.  ``flush``: end the accumulation window here (the last batch of an epoch)."""
        accumulate, step = self._window_phase(flush)
        losses, gflat = self._fwd_bwd(x_local, y_local, eps_local, accumulate=accumulate)
        self._bind_grads(gflat)
        if step:
            self._all_reduce(gflat)
            self._clip_norm(gflat)
            self.optimizer.step()
        self._end_micro_batch(step)
        return losses

    def _bind_grads(self, gflat: torch.Tensor) -> None:
        """Bind the .grad views of the trained parameters to the flat buffer: once, and again when the set of trained parameters changes
        (unfreezing the VAE after a classifier-only stage)."""
        trained = tuple(p.requires_grad for p, _ in self.hot.arena.entries)
        if self._views_of is not gflat or trained != self._views_trained:
            for (p, _), v in zip(self.hot.arena.entries, self.hot.arena.grad_views(gflat)):
                p.grad = v if p.requires_grad else None
            self._views_of = gflat
            self._views_trained = trained

    def _window_phase(self, flush: bool = False) -> Tuple[bool, bool]:
        """(accumulate, step) of the next micro-batch: does it add to the gradient buffer, does it end the window."""
        return self._micro > 0, bool(flush) or self._micro + 1 >= self.accumulate_grad_batches

    def _end_micro_batch(self, step: bool) -> None:
        self._micro = 0 if step else self._micro + 1

    def _knob_buffers(self, dev: torch.device) -> None:
        """The device buffers the options need, allocated before any capture (a CUDA graph must not own them)."""
        n = self.hot.arena.numel
        if self.accumulate_grad_batches > 1 and (self._acc_scratch is None or self._acc_scratch.device != dev):
            self._acc_scratch = torch.empty(n, dtype=torch.float32, device=dev)
        if self.gradient_clip_val is not None and self.gradient_clip_algorithm == "norm" and (self._norm_scratch is None or self._norm_scratch.device != dev):
            self._norm_scratch = torch.zeros(L.GRAD_NORM_SCRATCH_BYTES // 8, dtype=torch.float64, device=dev)
            self.grad_norm = torch.zeros((), dtype=torch.float32, device=dev)
            self._clip_coef = torch.ones((), dtype=torch.float32, device=dev)
            self.optimizer.clip_coef = self._clip_coef

    def _norm_spans(self):
        """The merged [a, b) spans the optimiser's update covers (FusedAdam._ranges over every group), as psvae_grad_norm takes them."""
        opt = self.optimizer
        spans = [(opt._offsets[id(p)], opt._offsets[id(p)] + p.numel()) for g in opt.param_groups for p in g["params"] if p.grad is not None]
        merged = opt._ranges(spans)
        if len(merged) > L.GRAD_NORM_MAX_SPANS:
            raise NotImplementedError(f"norm clipping covers at most {L.GRAD_NORM_MAX_SPANS} disjoint gradient spans, got {len(merged)}")
        return merged

    def _clip_norm(self, gflat: torch.Tensor) -> None:
        """Norm clipping: total norm and clip coefficient of the gradient the Adam pass is about to read (no host synchronisation)."""
        if self.gradient_clip_val is None or self.gradient_clip_algorithm != "norm":
            return
        from .engine import _on, _stream_ptr
        dev = gflat.device
        self._knob_buffers(dev)
        spans = self._norm_spans()
        flat = (C.c_int64 * (2 * len(spans)))(*[v for ab in spans for v in ab])
        with _on(dev):
            rc = L.lib().psvae_grad_norm(gflat.data_ptr(), flat, len(spans), float(self.optimizer.grad_scale), float(self.gradient_clip_val),
                                         self.grad_norm.data_ptr(), self._clip_coef.data_ptr(), self._norm_scratch.data_ptr(),
                                         self._norm_scratch.numel() * 8, _stream_ptr(dev))
        L.check(rc, "psvae_grad_norm")

    def _fwd_bwd(self, x_local: torch.Tensor, y_local=None, eps_local: Optional[torch.Tensor] = None, counters: Optional[torch.Tensor] = None,
                 accumulate: bool = False):
        """The fused forward + backward of train_step into the gradient buffer the all-reduce reads.  ``counters``: see HotPath.step.
        ``accumulate``: add to the buffer instead of overwriting it (a later micro-batch of an accumulation window)."""
        m, hot = self.module, self.hot
        gflat = self.symm.buf if self.symm is not None else (hot.arena.stage_buffer() if self._views_of is None else self._views_of)
        cons = getattr(m, "consistency_classifier", None)
        if accumulate:
            self._knob_buffers(gflat.device)
        losses, gflat, _ = hot.step(x_local, y_local if m.classifier is not None else None, eps_local, kl_weight=m.kl_loss_weight,
                                    clf_weight=m.classifier_loss_weight, use_cos_loss=m.use_cos_loss, compute_grads=True, grads=gflat,
                                    consistency=cons, consistency_y=y_local if cons is not None else None,
                                    consistency_weight=m.consitency_loss_weight, counters=counters, accumulate=accumulate,
                                    grad_scratch=self._acc_scratch if accumulate else None, grad_scope=hot.train_scope())
        return losses, gflat

    def _all_reduce(self, gflat: torch.Tensor, kind: Optional[str] = None) -> None:
        """The gradient all-reduce; ``kind`` overrides the symmetric-memory kind ``pick()`` chose (a CUDA graph may need NCCL).
        With a frozen VAE (classifier scope) only the classifier's span is reduced, with NCCL whatever kind was picked: the symmetric-memory
        kernels reduce the whole 5 MB buffer, the span is a few hundred bytes.  ``allreduce_kind`` then reads "nccl"; a full-scope step sets
        it back to the picked kind."""
        if self.world_size == 1 or self.local_only:
            return
        if self.hot.train_scope() == "classifier":
            a, b = self.hot.classifier_span()
            all_reduce_flat(gflat[a:b], self.bucket_bytes, self.group)
            self.allreduce_kind = "nccl"
        elif self.symm is not None:
            self.symm._call(kind or self.symm.kind)
            self.allreduce_kind = self.symm.kind
        else:
            all_reduce_flat(gflat, self.bucket_bytes, self.group)


def verify_data_parallel_step(device, steps: int = 3, global_batch: int = 8192, input_dim: int = 256, latent_dim: int = 64, num_classes: int = 2,
                              precision: str = "fp32", seed: int = 4321, group=None) -> dict:
    """Numerical self-check of the data-parallel path on the ranks that are actually running (what ``DDPStrategy`` guarantees for the
    reference, ps_vae/training.py:78): ``steps`` optimiser steps through ``DataParallelTrainer`` on this rank's shard of a seeded global
    batch with injected eps, then

      * every rank must hold BIT-identical parameters (all-gather of the flat buffer's checksum and of a strided sample), and
      * they must equal a single-process run on the whole global batch from the same initial parameters
        (``||p_dp - p_1|| / ||p_1||`` over the flat parameter buffer; gradients of the last step likewise).

    Runs in the deterministic summation mode (ordered split-K / bias sums) so that the only difference between the two runs is the
    grouping of fp32 partial sums.  Collective: call on every rank.  Returns the measured errors (rank 0 decides what to do with them)."""
    from . import _lib as L
    from .lightning import PseudoSpeakerVAE

    rank, ws = world()
    dev = torch.device(device)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(steps, global_batch, input_dim, generator=g)
    x = x / x.norm(dim=2, keepdim=True)
    y = torch.randint(0, num_classes, (steps, global_batch), generator=g)
    eps = torch.randn(steps, global_batch, latent_dim, generator=g)
    hp = dict(model=dict(input_dim=input_dim, latent_dim=latent_dim), classifier=dict(input_dim=latent_dim, num_classes=num_classes),
              optimizer=dict(lr=1e-3), scheduler=dict(T_max=200), precision=precision)
    prev = L.get_option("deterministic")
    L.set_option("deterministic", 1)
    try:
        torch.manual_seed(seed)                     # same initial weights on every rank and in the single-process twin
        dp = PseudoSpeakerVAE(**hp).to(dev)
        torch.manual_seed(seed)
        one = PseudoSpeakerVAE(**hp).to(dev)
        tr = DataParallelTrainer(dp, group=group)
        row0, rows = tr.set_shard(global_batch)
        solo = DataParallelTrainer(one, local_only=True)           # the twin: same three device-side calls, world of one, no collective
        for s in range(steps):
            xs, ys, es = (t[s].to(dev) for t in (x, y, eps))
            tr.train_step(xs[row0:row0 + rows], ys[row0:row0 + rows], es[row0:row0 + rows])
            solo.hot.row0 = 0
            solo.train_step(xs, ys, es)
        p_dp = dp.hot_path.arena.flat.detach().double()
        p_1 = one.hot_path.arena.flat.detach().double()
        g_dp = dp.hot_path.arena.flat_grad().detach().double() / ws       # the all-reduced SUM over ranks
        g_1 = one.hot_path.arena.flat_grad().detach().double()
        out = dict(world_size=ws, steps=steps, global_batch=global_batch, precision=precision,
                   param_rel_err=float((p_dp - p_1).norm() / p_1.norm()), grad_rel_err=float((g_dp - g_1).norm() / g_1.norm()),
                   param_max_abs=float((p_dp - p_1).abs().max()))
        flat32 = dp.hot_path.arena.flat.detach()
        sig = torch.cat([flat32.view(torch.int32).sum(dtype=torch.int64).reshape(1), flat32.view(torch.int32)[::997].to(torch.int64)])
        if ws > 1:
            sigs = [torch.empty_like(sig) for _ in range(ws)]
            dist.all_gather(sigs, sig, group=group)
            out["ranks_identical"] = bool(all(torch.equal(s, sigs[0]) for s in sigs))
        else:
            out["ranks_identical"] = True
        return out
    finally:
        L.set_option("deterministic", prev)
