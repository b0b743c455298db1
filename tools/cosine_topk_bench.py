"""Cosine top-k search (psvae_cosine_topk) on one GPU: time per shape with CUDA events after a warm-up call, the rate 2 Nq Nk D / t and
its share of the 2,250 TFLOP/s dense bf16 data-sheet figure, the bf16 selection error at D = 256, and a torch bf16 chunked mm + topk
baseline at 1,048,576 x 674,068 with its index agreement.  The GPU name and power limit are read in the same run.

    python tools/cosine_topk_bench.py --out profiles/r07_cosine_topk.txt [--quick]

Inputs are seeded Gaussian fp32 rows (12.5 M x 256 fp32 queries: 12.8 GB; 674,068 keys: 0.69 GB, larger than the 126 MB L2)."""
import argparse
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_BF16 = 2250e12
DEV = "cuda:0"


def gpu_facts():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # pragma: no cover
        return f"nvidia-smi unavailable ({e})"


def data(n, d, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(n, d, generator=g, device=DEV)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        out = fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / 1e3 / reps, out


def torch_baseline(q, x, k, chunk=8192):
    qb = torch.nn.functional.normalize(q, dim=1).to(torch.bfloat16)
    xb = torch.nn.functional.normalize(x, dim=1).to(torch.bfloat16)
    sims, idxs = [], []
    for a in range(0, q.shape[0], chunk):
        s = torch.mm(qb[a:a + chunk], xb.T)
        v, i = torch.topk(s, k, dim=1)
        sims.append(v)
        idxs.append(i)
    return torch.cat(sims), torch.cat(idxs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_cosine_topk.txt"))
    ap.add_argument("--quick", action="store_true", help="only the 1 M-query shapes and the baseline")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU only")
    import pseudo_speaker_vae_b200 as P

    torch.backends.cuda.matmul.allow_tf32 = False
    lines = [f"# cosine top-k search (psvae_cosine_topk), tools/cosine_topk_bench.py", f"# GPU: {gpu_facts()}",
             "# time: CUDA events around whole cosine_topk calls (normalisation + search + merge/re-rank, chunks of 1,048,576 queries) after"
             " one warm-up call; rate = 2 Nq Nk D / t; share = rate / 2,250 TFLOP/s (dense bf16 data sheet, 1,000 W)"]

    # bf16 selection error at D = 256: scores of bf16-rounded unit vectors (fp32 accumulation) against fp64
    q = data(4096, 256, 1)
    x = data(65536, 256, 2)
    uq, ux = torch.nn.functional.normalize(q.double(), dim=1), torch.nn.functional.normalize(x.double(), dim=1)
    exact = uq @ ux.T
    sel = uq.float().to(torch.bfloat16).float() @ ux.float().to(torch.bfloat16).float().T
    err = (sel.double() - exact).abs()
    lines.append(f"bf16 selection error at D=256 (4,096 x 65,536 Gaussian pairs): max {err.max().item():.3e}, "
                 f"99.9th percentile {torch.quantile(err.flatten()[:1 << 24].float(), 0.999).item():.3e}")
    del q, x, uq, ux, exact, sel, err

    shapes = [(1048576, 674068, 256, 1), (1048576, 674068, 256, 16)]
    if not args.quick:
        shapes += [(12500000, 674068, 256, 1), (12500000, 674068, 256, 16), (10000, 12500000, 256, 1), (1048576, 674068, 512, 16)]
    lines.append(f"{'Nq':>10} {'Nk':>10} {'D':>4} {'k':>3} {'time s':>9} {'TFLOP/s':>9} {'share':>7}")
    for nq, nk, d, k in shapes:
        q = data(nq, d, 3)
        x = data(nk, d, 4)
        reps = 3 if nq * nk <= 1048576 * 674068 else 1
        t, _ = timed(lambda: P.cosine_topk(q, x, k), reps)
        rate = 2.0 * nq * nk * d / t
        lines.append(f"{nq:>10,} {nk:>10,} {d:>4} {k:>3} {t:>9.4f} {rate / 1e12:>9.1f} {rate / PEAK_BF16:>7.1%}")
        print(lines[-1], flush=True)
        del q, x
        torch.cuda.empty_cache()

    # torch baseline: chunked bf16 mm + topk (the similarity matrix is written and read back chunk by chunk)
    nq, nk, d = 1048576, 674068, 256
    q = data(nq, d, 3)
    x = data(nk, d, 4)
    t0, (ts, ti) = timed(lambda: torch_baseline(q, x, 1), 1)
    t1, (s1, i1) = timed(lambda: P.cosine_topk(q, x, 1), 1)
    agree = (ti[:, 0] == i1[:, 0]).float().mean().item()
    # rows where the exact top-1 and top-2 (fp32 re-scored by cosine_topk at k = 2) are more than 2 x 2^-8 apart: the baseline's bf16 output
    # rounding cannot reorder them
    s2, i2 = P.cosine_topk(q, x, 2)
    sep = (s2[:, 0] - s2[:, 1]) > 2 * 2.0 ** -7
    agree_sep = (ti[sep, 0] == i1[sep, 0]).float().mean().item()
    lines.append(f"torch bf16 chunked mm + topk, {nq:,} x {nk:,}, D={d}, k=1: {t0:.3f} s ({2.0 * nq * nk * d / t0 / 1e12:.1f} TFLOP/s); "
                 f"cosine_topk {t1:.3f} s; indices agree on {agree:.4%} of rows, on {agree_sep:.4%} of the {sep.float().mean().item():.1%} rows "
                 f"whose top-2 gap exceeds 2^-6 (the baseline rounds its scores to bf16: ties and swaps below that)")
    print("\n".join(lines))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    t = time.time()
    main()
    print(f"total {time.time() - t:.0f} s")
