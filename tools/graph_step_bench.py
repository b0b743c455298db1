"""Eager vs CUDA-graph train step (pseudo_speaker_vae_b200.GraphedTrainStep) across batch sizes, bf16, the benchmark's model (D = 256, L = 64,
2-class linear classifier), one GPU.  For each B:

  eager_ms        DataParallelTrainer.train_step, CUDA events over --steps steps after --warmup steps
  enqueue_us      host time to enqueue one eager step (perf_counter around 20 calls issued right after a synchronise, no sync inside:
                  the launch queue never fills, so this is what the host spends per step, not what the GPU does)
  graph_ms        GraphedTrainStep replays, CUDA events over --steps steps after --warmup calls (call 1 eager, call 2 captures)

plus an end-to-end leg at B = 2,048: PinnedBatchLoader over a pinned bf16 store -> step, eager and graphed (the batch is copied into the
graph's static buffer).  Four distinct input batches rotate.  The GPU's name and power limit are read in the same run.

    python tools/graph_step_bench.py [--sizes 256,1024,2048,8192,65536] [--steps 200] [--warmup 50] [--out FILE.json]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import pseudo_speaker_vae_b200 as P  # noqa: E402
from pseudo_speaker_vae_b200 import _lib as L  # noqa: E402
from pseudo_speaker_vae_b200 import data as PD  # noqa: E402

D, LAT, NB = 256, 64, 4


def gpu_info():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e!r})"
    return info


def make(B, seed=0):
    torch.manual_seed(seed)
    m = P.PseudoSpeakerVAE(model=dict(input_dim=D, latent_dim=LAT), classifier=dict(input_dim=LAT, num_classes=2), optimizer=dict(lr=1e-3),
                           scheduler=dict(T_max=200), precision="bf16").to("cuda")
    m.hot_path.manual_seed(1236, 0)
    return m, P.DataParallelTrainer(m, local_only=True)


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


def one_size(B, steps, warmup):
    bs = batches(B)
    _, tr = make(B)
    run = lambda i: tr.train_step(*bs[i % NB])
    for i in range(warmup):
        run(i)
    eager_ms = timed(run, steps)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(20):
        run(i)
    enqueue_us = (time.perf_counter() - t0) / 20 * 1e6
    torch.cuda.synchronize()
    _, trg = make(B)
    gs = P.GraphedTrainStep(trg, rows=B, x_dtype=torch.bfloat16)
    rung = lambda i: gs(*bs[i % NB])
    for i in range(warmup):
        rung(i)
    graph_ms = timed(rung, steps)
    return dict(B=B, eager_ms=eager_ms, enqueue_us=enqueue_us, graph_ms=graph_ms, speedup=eager_ms / graph_ms, pdl_in_graph=gs.pdl,
                replays=gs.replays)


def loader_leg(B, steps, warmup):
    g = torch.Generator().manual_seed(7)
    n = NB * B
    x = torch.randn(n, D, generator=g)
    x = (x / x.norm(dim=1, keepdim=True)).numpy()
    y = torch.randint(0, 2, (n,), generator=g).numpy().astype(np.int64)
    tmp = tempfile.mkdtemp(prefix="psvae_graph_bench_")
    store = PD.PackedEmbeddingStore.from_arrays(tmp, x, y, ["gender"], dtype="bf16")
    store.pin()
    out = dict(B=B)
    for name in ("eager", "graph"):
        _, tr = make(B)
        step = P.GraphedTrainStep(tr, rows=B, x_dtype=torch.bfloat16) if name == "graph" else tr.train_step
        loader = PD.PinnedBatchLoader(store, B, device="cuda", shuffle=False, seed=3)

        def run_n(k):
            done = 0
            while done < k:
                for xb, yb in loader:
                    step(xb, yb)
                    done += 1
                    if done >= k:
                        break
        run_n(warmup)
        out[f"{name}_ms"] = _timed_block(run_n, steps)
    out["speedup"] = out["eager_ms"] / out["graph_ms"]
    del store
    shutil.rmtree(tmp, ignore_errors=True)
    return out


def _timed_block(run_n, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    run_n(steps)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="256,1024,2048,8192,65536")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the GPU and has no CPU mode")
    res = dict(gpu=gpu_info(), steps=args.steps, warmup=args.warmup, options=dict(deterministic=L.get_option("deterministic"), pdl=L.get_option("pdl")),
               sizes=[])
    print(json.dumps(res["gpu"]), flush=True)
    print(f"{'B':>7} {'eager ms':>9} {'enqueue us':>11} {'graph ms':>9} {'speedup':>8}", flush=True)
    for B in [int(s) for s in args.sizes.split(",")]:
        r = one_size(B, args.steps, args.warmup)
        res["sizes"].append(r)
        print(f"{B:>7} {r['eager_ms']:>9.4f} {r['enqueue_us']:>11.1f} {r['graph_ms']:>9.4f} {r['speedup']:>8.3f}", flush=True)
    r = loader_leg(2048, args.steps, args.warmup)
    res["loader_2048"] = r
    print(f"PinnedBatchLoader leg B=2048: eager {r['eager_ms']:.4f} ms/step, graphed {r['graph_ms']:.4f} ms/step ({r['speedup']:.3f}x)", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
