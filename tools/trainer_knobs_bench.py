"""Cost of the trainer options (gradient clipping, gradient accumulation) on the benchmark's model (bf16, D = 256, L = 64, hidden 512x2,
2-class linear classifier), one GPU, CUDA events after warm-up.  All times are per OPTIMISER step.

  clip       graphed B = 2,048 and eager B = 65,536: no clipping / norm clipping / value clipping
  accumulate eager 4 x 16,384 vs 1 x 65,536 and graphed 4 x 512 vs 1 x 2,048 (same rows per optimiser step)
  norm pass  psvae_grad_norm alone on the 5.13 MB gradient buffer (events around --steps back-to-back launches)
  launches   psvae_launch_count per optimiser step of the eager path, per configuration

The GPU's name, power limit and max SM clock are read (nvidia-smi, read-only query) in the same run.

    python tools/trainer_knobs_bench.py [--steps 200] [--warmup 50] [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import pseudo_speaker_vae_b200 as P  # noqa: E402
from pseudo_speaker_vae_b200 import _lib as L  # noqa: E402
from pseudo_speaker_vae_b200.engine import _stream_ptr  # noqa: E402

D, LAT, NB = 256, 64, 4
CLIPS = {"none": {}, "norm": dict(gradient_clip_val=1.0), "value": dict(gradient_clip_val=1e-3, gradient_clip_algorithm="value")}


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e!r})"


def make(k=1, **knobs):
    torch.manual_seed(0)
    m = P.PseudoSpeakerVAE(model=dict(input_dim=D, latent_dim=LAT), classifier=dict(input_dim=LAT, num_classes=2), optimizer=dict(lr=1e-3),
                           scheduler=dict(T_max=200), precision="bf16").to("cuda")
    m.hot_path.manual_seed(1236, 0)
    return P.DataParallelTrainer(m, local_only=True, accumulate_grad_batches=k, **knobs)


def batches(B):
    g = torch.Generator().manual_seed(1234)
    out = []
    for _ in range(NB):
        x = torch.randn(B, D, generator=g)
        x = x / x.norm(dim=1, keepdim=True)
        out.append((x.to(torch.bfloat16).cuda(), torch.randint(0, 2, (B,), generator=g).cuda()))
    return out


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def per_opt_step(B, k, graphed, steps, warmup, **knobs):
    """ms per optimiser step (k micro-batches of B rows) and, eager, the library launches per optimiser step."""
    bs = batches(B)
    tr = make(k, **knobs)
    step = P.GraphedTrainStep(tr, rows=B, x_dtype=torch.bfloat16) if graphed else tr.train_step
    run = lambda i: step(*bs[i % NB])
    for i in range(warmup * k):
        run(i)
    ms = timed(run, steps * k) * k
    n0 = int(L.lib().psvae_launch_count())
    for i in range(k):
        run(i)
    torch.cuda.synchronize()
    return ms, int(L.lib().psvae_launch_count()) - n0


def norm_pass(steps, warmup):
    tr = make(1, gradient_clip_val=1.0)
    x, y = batches(2048)[0]
    tr.train_step(x, y)
    g = tr.hot.arena.flat_grad()
    spans = tr._norm_spans()
    flat = (C.c_int64 * (2 * len(spans)))(*[v for ab in spans for v in ab])
    lib, st = L.lib(), _stream_ptr(g.device)
    call = lambda i: L.check(lib.psvae_grad_norm(g.data_ptr(), flat, len(spans), 1.0, 1.0, tr.grad_norm.data_ptr(), tr._clip_coef.data_ptr(),
                                                 tr._norm_scratch.data_ptr(), tr._norm_scratch.numel() * 8, st))
    for i in range(warmup):
        call(i)
    return timed(call, steps) * 1e3, g.numel() * 4, len(spans)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the GPU and has no CPU mode")
    res = dict(gpu=gpu_info(), steps=args.steps, warmup=args.warmup, options=dict(deterministic=L.get_option("deterministic"), pdl=L.get_option("pdl")))
    print("# GPU (name, power limit, max SM clock): " + res["gpu"], flush=True)
    print(f"# bf16 D={D} L={LAT}, fast summation mode, pdl={res['options']['pdl']}; CUDA events over {args.steps} optimiser steps after "
          f"{args.warmup} warm-up steps; ms per optimiser step", flush=True)
    res["clip"] = {}
    print(f"{'path':>18} {'clip':>6} {'ms/step':>9} {'launches':>9}", flush=True)
    for B, graphed in ((2048, True), (65536, False)):
        for name, kw in CLIPS.items():
            ms, launches = per_opt_step(B, 1, graphed, args.steps, args.warmup, **kw)
            res["clip"][f"{'graph' if graphed else 'eager'}_{B}_{name}"] = dict(ms=ms, launches_eager=None if graphed else launches)
            print(f"{('graph' if graphed else 'eager') + ' B=' + str(B):>18} {name:>6} {ms:>9.4f} {'-' if graphed else launches:>9}", flush=True)
    res["accumulate"] = {}
    print(f"{'path':>18} {'k x B':>12} {'ms/step':>9} {'launches':>9}", flush=True)
    for graphed, pairs in ((False, ((1, 65536), (4, 16384))), (True, ((1, 2048), (4, 512)))):
        for k, B in pairs:
            ms, launches = per_opt_step(B, k, graphed, args.steps, args.warmup)
            res["accumulate"][f"{'graph' if graphed else 'eager'}_{k}x{B}"] = dict(ms=ms, launches=launches)
            print(f"{'graph' if graphed else 'eager':>18} {f'{k} x {B}':>12} {ms:>9.4f} {launches:>9}", flush=True)
    us, nbytes, nspans = norm_pass(args.steps * 10, args.warmup)
    res["norm_pass"] = dict(us=us, bytes=nbytes, spans=nspans, gb_per_s=nbytes / us * 1e-3)
    print(f"psvae_grad_norm alone: {us:.2f} us over {nbytes / 1e6:.2f} MB in {nspans} span(s) = {nbytes / us * 1e-3:.0f} GB/s "
          f"(back-to-back launches: the gradient stays in L2)", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
