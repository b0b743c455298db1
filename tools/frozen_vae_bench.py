"""Full train step against the classifier-only step (frozen VAE, freeze_vae) on the benchmark's model (bf16 fast mode, D = 256, L = 64,
hidden 512x2, 2-class linear classifier), one GPU, CUDA events after warm-up.  Per optimiser step:

  eager      B = 65,536   DataParallelTrainer.train_step
  graphed    B = 2,048    GraphedTrainStep
  lightning  B = 2,048    training_step -> loss.backward() -> FusedAdam.step()

Each leg alternates full / frozen for --repeats rounds (the spread shows in the per-round numbers) and counts psvae_launch_count per
step.  `rows_kernel` compares the two ways of forming the classifier's gradient under the fused encoder head at B = 65,536: the fused head
plus clf_rows_wgrad_kernel (the default), against the same step with option fused_head = 0 (grouped head GEMM + the fused classifier pass,
which writes the gradient itself); `profile` is the kernel time of clf_rows_wgrad_kernel from torch.profiler, in a run of its own.
The GPU's name, power limit and max SM clock are read (nvidia-smi, read-only query) in the same run.

    python tools/frozen_vae_bench.py [--steps 100] [--warmup 20] [--repeats 3] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import pseudo_speaker_vae_b200 as P  # noqa: E402
from pseudo_speaker_vae_b200 import _lib as L  # noqa: E402

D, LAT, NB = 256, 64, 4


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e!r})"


def make(frozen):
    torch.manual_seed(0)
    m = P.PseudoSpeakerVAE(model=dict(input_dim=D, latent_dim=LAT), classifier=dict(input_dim=LAT, num_classes=2), optimizer=dict(lr=1e-3),
                           scheduler=dict(T_max=200), precision="bf16", freeze_vae=frozen).to("cuda")
    m.hot_path.manual_seed(1236, 0)
    return m


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


def launches(fn):
    c0 = L.lib().psvae_launch_count()
    fn(0)
    torch.cuda.synchronize()
    return int(L.lib().psvae_launch_count() - c0)


def leg(kind, frozen, B):
    data = batches(B)
    m = make(frozen)
    if kind == "lightning":
        opt = m.configure_optimizers()["optimizer"]

        def fn(i):
            x, y = data[i % NB]
            m.training_step((x, y), i)["loss"].backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
        return fn
    tr = P.DataParallelTrainer(m, local_only=True)
    if kind == "graphed":
        step = P.GraphedTrainStep(tr, rows=B)
        return lambda i: step(*data[i % NB])
    return lambda i: tr.train_step(*data[i % NB])


def profile_rows_kernel(B):
    m = make(True)
    tr = P.DataParallelTrainer(m, local_only=True)
    data = batches(B)
    for i in range(5):
        tr.train_step(*data[i % NB])
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(20):
            tr.train_step(*data[i % NB])
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.count >= 20:
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            out[ev.key[:90]] = round(t / ev.count, 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("frozen_vae_bench needs a CUDA device")
    L.set_option("deterministic", 0)
    res = dict(gpu=gpu_info(), precision="bf16 fast", steps=a.steps, warmup=a.warmup, legs={})
    for kind, B in (("eager", 65536), ("graphed", 2048), ("lightning", 2048)):
        fns = {name: leg(kind, name == "frozen", B) for name in ("full", "frozen")}
        for fn in fns.values():
            for i in range(a.warmup):
                fn(i)
        torch.cuda.synchronize()
        r = {name: dict(ms=[]) for name in fns}
        for _ in range(a.repeats):                       # alternating A/B rounds
            for name, fn in fns.items():
                r[name]["ms"].append(round(timed(fn, a.steps), 4))
        for name, fn in fns.items():
            r[name]["launches_per_step"] = launches(fn)
            r[name]["ms_median"] = sorted(r[name]["ms"])[len(r[name]["ms"]) // 2]
        r["speedup"] = round(r["full"]["ms_median"] / r["frozen"]["ms_median"], 2)
        res["legs"][f"{kind}_B{B}"] = r
        print(kind, B, json.dumps(r), flush=True)
    # the fused head + row-gradient kernel against the unfused forward whose classifier pass writes the gradient itself
    rk = {}
    for fh in (1, 0):
        L.set_option("fused_head", fh)
        fn = leg("eager", True, 65536)
        for i in range(a.warmup):
            fn(i)
        rk[f"fused_head={fh}"] = [round(timed(fn, a.steps), 4) for _ in range(a.repeats)]
    L.set_option("fused_head", 1)
    res["rows_kernel"] = rk
    print("rows_kernel", json.dumps(rk), flush=True)
    try:
        res["profile_us_per_launch"] = profile_rows_kernel(65536)
    except Exception as e:  # noqa: BLE001 -- the timings above stand without it
        res["profile_us_per_launch"] = repr(e)
    print("profile", json.dumps(res["profile_us_per_launch"]), flush=True)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
