"""Conditional sampling with one target for the batch against per-row targets and an in-kernel target mix: N samples x STEPS Langevin
steps plus the decode, through sample_on_device, the three forms alternating in each round.  Two classifiers: two linear heads on z
(gender 3 + age 3: the thread-per-sample kernel) and BASELINE config 4's 2-layer multi-label classifier, hidden 128 (the generic kernel).

    python tools/langevin_bench.py [--n 12500000] [--steps 100] [--rounds 3] [--targets shared,rows,mix]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pseudo_speaker_vae_b200 as P  # noqa: E402

HEADS = {"gender": 3, "age": 3}
MIX = [({"gender": 0, "age": 0}, 0.2), ({"gender": 0, "age": 2}, 0.3), ({"gender": 1, "age": 1}, 0.4), ({"gender": 1}, 0.1)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=12_500_000, help="samples per call (BASELINE config 4: 100 M over 8 GPUs)")
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--targets", default="shared,rows,mix", help="comma list of shared | rows | mix")
    args = ap.parse_args()
    forms = args.targets.split(",")
    if not set(forms) <= {"shared", "rows", "mix"}:
        raise SystemExit(f"--targets: unknown form in {args.targets!r}")
    N, STEPS = args.n, args.steps
    print(f"GPU: {gpu_info()}")
    print(f"N = {N:,} samples x {STEPS} Langevin steps + decode (D = 256, L = 64, bf16), ms per call from CUDA events; forms alternate in each round")
    out = torch.empty(N, 256, dtype=torch.float32, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    rows = {"gender": torch.randint(0, 2, (N,), device="cuda", generator=g), "age": torch.randint(0, 3, (N,), device="cuda", generator=g)}
    for kind in ("linear heads (fast kernel)", "config 4 MLP classifier, 2 layers, hidden 128 (generic kernel)"):
        torch.manual_seed(0)
        clf = dict(input_dim=64, num_classes=dict(HEADS))
        if kind.startswith("config 4"):
            clf.update(num_layers=2, hidden_dim=128)
        m = P.PseudoSpeakerVAE(model=dict(input_dim=256, latent_dim=64), classifier=clf, optimizer={}, scheduler=dict(T_max=1),
                               precision="bf16").to("cuda")
        calls = {
            "shared": lambda: P.sample_on_device(m, N, {"gender": 1, "age": 1}, num_steps=STEPS, out=out),
            "rows": lambda: P.sample_on_device(m, N, rows, num_steps=STEPS, out=out),
            "mix": lambda: P.sample_on_device(m, N, num_steps=STEPS, out=out, target_mix=MIX),
        }
        for f in forms:                                       # warm-up: module load, smem attributes, the decode workspace
            calls[f]()
        torch.cuda.synchronize()
        ms = {f: [] for f in forms}
        for _ in range(args.rounds):
            for f in forms:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                calls[f]()
                e1.record()
                torch.cuda.synchronize()
                ms[f].append(round(e0.elapsed_time(e1), 2))
        print(f"\n{kind}")
        base = sorted(ms[forms[0]])[len(ms[forms[0]]) // 2]
        for f in forms:
            med = sorted(ms[f])[len(ms[f]) // 2]
            print(f"  {f:7s} ms {ms[f]}  median {med:.2f}  {N / med / 1e3:.2f} M samples/s  median / {forms[0]} {med / base:.4f}")
    print(f"\nGPU (after): {gpu_info()}")


if __name__ == "__main__":
    main()
