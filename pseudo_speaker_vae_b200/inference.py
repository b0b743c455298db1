"""Sampling: drop-ins for ``unconditional_synthesis`` / ``conditional_synthesis`` of ps_vae/inference.py:10-110
and the CLI of :113-156.

Same signatures and return values (CPU tensors; ``(x_hat, history)`` with ``return_history=True`` where
``history`` is a list of ``num_steps`` numpy arrays ``[N, latent]``).  Underneath:

  * unconditional: z ~ N(0, I) is drawn by the library's counter-based Philox generator inside the decode call
    (counter = global sample index, so a sharded run reproduces the single-GPU batch bit for bit) and goes through
    the decoder GEMM chain;
  * conditional: the whole Langevin loop (inference.py:77-103) is ONE kernel launch -- closed-form classifier
    gradient, in-kernel noise, no host round trips (the reference does a D2H copy of z plus two ``.item()`` syncs
    every step, SURVEY F12); the z history is materialised only when asked for.

``sample_on_device`` is the bulk path (BASELINE config 4): it writes into a caller-provided device buffer and
returns without synchronising, and ``shard_rows`` gives each data-parallel rank its slice of the sample index range.

Conditioning: ``classifier_target`` is one target for the batch (an int, or a dict of label -> class) or one per row (a length-N integer
tensor, or a dict whose values are ints or length-N integer tensors; -1 leaves a head out for that row).  ``target_mix=[(target, weight),
...]`` instead draws every row's target in the kernel from its global row index, so a population with a demographic mix comes out of one
call, and a sharded run draws the same targets as a single call.  Every row is bit-identical to a shared-target call with that row's target.
"""
from __future__ import annotations

import argparse
import os
from typing import List, Optional, Tuple, Union

import torch
from torch import Tensor

from .utils import parse_classifier_target, parse_target_mix, sample_filename


def _hot(vae_model):
    hot = getattr(vae_model, "hot_path", None)
    if hot is None:
        raise TypeError("vae_model must be a pseudo_speaker_vae_b200 PseudoSpeakerVAE / VAEModel")
    return hot() if callable(hot) else hot


def _check_device(vae_model, device) -> None:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"device={device!r}: pseudo_speaker_vae_b200 samples on a CUDA (B200) device only; there is no CPU fallback")
    mdev = _hot(vae_model).arena.device
    if mdev.type != "cuda" or (dev.index is not None and mdev.index != dev.index):
        raise RuntimeError(f"the model lives on {mdev} but device={device!r} was requested; move the model first (model.to(device))")


def shard_rows(num_samples: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous slice [row0, row0 + rows) of the global sample index range owned by ``rank`` (SURVEY 8(e))."""
    base, rem = divmod(int(num_samples), int(world_size))
    rows = base + (1 if rank < rem else 0)
    row0 = rank * base + min(rank, rem)
    return row0, rows


def sample_on_device(vae_model, num_samples: int, classifier_target=None, step_size: float = 0.01, num_steps: int = 100,
                     noise_weight: float = 1.0, out: Optional[Tensor] = None, row0: int = 0, *, target_mix=None):
    """Generate ``num_samples`` embeddings into ``out`` (device tensor) without any host synchronisation.

    ``row0`` is the global index of the first sample: rank r of a sharded run passes ``shard_rows(N, r, W)``.  Per-row targets are not
    validated on the host (that would synchronise): a row with a target out of range comes out as NaN.  With ``target_mix`` the result is
    ``(out, targets)``, the drawn targets on the device: int64 ``[N]`` for a single-label classifier, else ``{label: int64 [N]}`` (-1: head
    left out)."""
    hot = _hot(vae_model)
    if classifier_target is None and target_mix is None:
        return hot.decode(None, num_samples=num_samples, out=out, row0=row0)
    res = hot.langevin(num_samples, classifier_target, step_size, num_steps, noise_weight, row0=row0, target_mix=target_mix)
    x = hot.decode(res[0], out=out)
    return (x, res[3]) if target_mix is not None else x


def unconditional_synthesis(vae_model, num_samples: int, device: str) -> Tensor:
    """z ~ N(0, I) -> decode -> CPU (inference.py:10-27)."""
    _check_device(vae_model, device)
    return _hot(vae_model).decode(None, num_samples=num_samples).detach().cpu()


def conditional_synthesis(vae_model, num_samples: int, classifier_target=None, step_size: float = 0.01, num_steps: int = 100,
                          noise_weight: float = 1.0, return_history: bool = False, device: str = "cpu", *, z0: Optional[Tensor] = None,
                          noise: Optional[Tensor] = None, target_mix=None):
    """Classifier-guided Langevin dynamics in latent space, then decode (inference.py:29-110).

    ``z0`` / ``noise`` (keyword-only, optional) inject the initial draw and the per-step noise ``[num_steps, N, latent]``
    for parity runs; by default both come from the in-kernel Philox generator.  ``classifier_target`` may be per row (checked on the host:
    IndexError / ValueError for a bad row).  With ``target_mix`` (and no ``classifier_target``) the drawn targets are returned last:
    ``(x_hat, targets)`` or ``(x_hat, history, targets)``, on the CPU in the form ``sample_on_device`` gives."""
    _check_device(vae_model, device)
    hot = _hot(vae_model)
    res = hot.langevin(num_samples, classifier_target, step_size, num_steps, noise_weight, z0=z0, noise=noise,
                       return_history=return_history, target_mix=target_mix, check_targets=True)
    z, hist = res[0], res[1]
    x_hat = hot.decode(z).detach().cpu()
    out = (x_hat,)
    if return_history:
        h = hist.cpu().numpy()
        history: List = [h[i] for i in range(h.shape[0])]
        out += (history,)
    if target_mix is not None:
        t = res[3]
        out += ({k: v.cpu() for k, v in t.items()} if isinstance(t, dict) else t.cpu(),)
    return out if len(out) > 1 else x_hat


def latent_transformation(vae_model, embeddings: Tensor, classifier_target: Union[int, dict], step_size: float = 0.02, max_steps: int = 10000,
                          noise_weight: float = 0.0, prior_weight: float = 0.5, threshold: float = 0.95, return_history: bool = False,
                          noise: Optional[Tensor] = None):
    """The attribute-transformation loop of analysis/sample_gender_transformation.py:57-99, batched: every embedding is encoded
    (``_, z, _ = vae_model(embed)``: z = the encoder mean), its latent ascends ``log p(y|z) + prior_weight * log p(z)`` with steps of
    ``0.5 * step_size**2`` (plus ``step_size * noise_weight * N(0, I)``) and is frozen after the update of the first step whose
    ``p(y|z)`` exceeded ``threshold`` -- one kernel launch for all samples and all steps instead of a Python loop with two ``.item()`` syncs per
    step.  Returns ``(x_hat [N, D] cpu, z [N, L] cpu, stop_step [N] cpu int32 (max_steps: never stopped), prob [N] cpu)``, plus the list of
    per-step latents with ``return_history``.  ``classifier_target`` may be per row (each speaker its own target, e.g. the opposite of
    its own gender; checked on the host)."""
    hot = _hot(vae_model)
    dev = hot.arena.device
    with torch.no_grad():
        _, mu, _ = hot.forward(embeddings.to(dev))
    z, hist, (_, stop, prob) = hot.langevin(mu.shape[0], classifier_target, step_size, max_steps, noise_weight, z0=mu, noise=noise,
                                             return_history=return_history, prior_weight=prior_weight, threshold=threshold, return_stop=True,
                                             check_targets=True)
    x_hat = hot.decode(z).detach().cpu()
    out = (x_hat, z.cpu(), stop.cpu(), prob.cpu())
    if return_history:
        h = hist.cpu().numpy()
        return out + ([h[i] for i in range(h.shape[0])],)
    return out


def _write_rows(rows: Tensor, first: int, save_dir: str) -> List[str]:
    paths = []
    for j in range(rows.shape[0]):
        path = os.path.join(save_dir, sample_filename(first + j))
        torch.save(rows[j].clone(), path)
        paths.append(path)
    return paths


def save_samples(x_hat: Tensor, save_dir: str, workers: int = 0, chunk: int = 4096) -> List[str]:
    """Row i -> ``sample_{i}.pt`` (inference.py:154-156), file contents identical to the reference's ``torch.save(x, path)``.

    The reference writes one file per row in a serial loop after the whole batch has been copied to the host.  Here a device batch is
    brought over in chunks of ``chunk`` rows on a copy stream into pinned memory while ``workers`` threads (default: 8, or 0 for the
    caller's thread when the batch is small) serialise the previous chunk -- the D2H copy, the pickling and the file system calls overlap."""
    os.makedirs(save_dir, exist_ok=True)
    n = int(x_hat.shape[0])
    if workers <= 0:
        workers = 8 if n >= 256 else 0
    if workers == 0 and not x_hat.is_cuda:
        return _write_rows(x_hat, 0, save_dir)
    from concurrent.futures import ThreadPoolExecutor

    futures = []
    with ThreadPoolExecutor(max_workers=max(1, workers)) as pool:
        if x_hat.is_cuda:
            stream = torch.cuda.Stream(x_hat.device)
            stream.wait_stream(torch.cuda.current_stream(x_hat.device))
            for a in range(0, n, chunk):
                b = min(n, a + chunk)
                host = torch.empty((b - a,) + tuple(x_hat.shape[1:]), dtype=x_hat.dtype, pin_memory=True)
                with torch.cuda.stream(stream):
                    host.copy_(x_hat[a:b], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(stream)

                def job(host=host, a=a, ev=ev):
                    ev.synchronize()
                    return _write_rows(host, a, save_dir)

                futures.append(pool.submit(job))
        else:
            per = max(1, -(-n // (4 * max(1, workers))))
            for a in range(0, n, per):
                futures.append(pool.submit(_write_rows, x_hat[a:a + per], a, save_dir))
        paths: List[str] = []
        for f in futures:
            paths += f.result()
    return paths


def main(argv=None) -> None:
    from .lightning import PseudoSpeakerVAE

    parser = argparse.ArgumentParser(description="Generate synthetic embeddings using a VAE model.")
    parser.add_argument("--vae_ckpt_path", type=str, required=True, help="Path to the VAE checkpoint.")
    parser.add_argument("--n_samples", type=int, default=16, help="Number of samples to generate.")
    parser.add_argument("--save_dir", type=str, required=True, help="Directory to save the generated samples.")
    parser.add_argument("--synthesis_type", type=str, choices=["conditional", "unconditional"], required=True)
    parser.add_argument("--classifier_target", type=str, default=None, help="Target class (int, or JSON dict for multi-label); default 1.")
    parser.add_argument("--target_mix", type=str, default=None,
                        help='Draw each sample\'s target from a weighted mix, JSON [[target, weight], ...], e.g. '
                             '\'[[{"gender": 0, "age": 1}, 0.3], [{"gender": 1, "age": 1}, 0.7]]\'; the drawn targets go to <save_dir>/targets.pt.')
    parser.add_argument("--num_steps", type=int, default=5000)
    parser.add_argument("--step_size", type=float, default=0.01)
    parser.add_argument("--noise_weight", type=float, default=1.0)
    parser.add_argument("--device", type=str, default="cuda", help="CUDA device (this implementation has no CPU path).")
    parser.add_argument("--nearest_store", type=str, default=None,
                        help="A PackedEmbeddingStore directory (e.g. the training set): each sample's nearest entries by cosine similarity, "
                             "computed on the device, go to <save_dir>/nearest.pt as {'index': int64 [N, k], 'similarity': float32 [N, k]}.")
    parser.add_argument("--nearest_k", type=int, default=1, help="Entries per sample for --nearest_store (1..16).")
    args = parser.parse_args(argv)
    if args.nearest_store is not None:
        if not 1 <= args.nearest_k <= 16:
            parser.error(f"--nearest_k must be in [1, 16], got {args.nearest_k}")
        if not os.path.isfile(os.path.join(args.nearest_store, "index.json")):
            parser.error(f"--nearest_store {args.nearest_store!r} is not a PackedEmbeddingStore (no index.json)")
    target_mix = None
    if args.target_mix is not None:
        if args.classifier_target is not None:
            parser.error("--target_mix and --classifier_target are mutually exclusive")
        if args.synthesis_type != "conditional":
            parser.error("--target_mix needs --synthesis_type conditional")
        try:
            target_mix = parse_target_mix(args.target_mix)
        except ValueError as e:
            parser.error(str(e))

    classifier_target = None if target_mix is not None else parse_classifier_target(args.classifier_target or "1")
    model = PseudoSpeakerVAE.load_from_checkpoint(args.vae_ckpt_path)
    model = model.to(args.device)
    targets = None
    if args.synthesis_type == "conditional":
        x_hat = conditional_synthesis(model, classifier_target=classifier_target, num_samples=args.n_samples, num_steps=args.num_steps,
                                      step_size=args.step_size, noise_weight=args.noise_weight, device=args.device, target_mix=target_mix)
        if target_mix is not None:
            x_hat, targets = x_hat
    else:
        x_hat = unconditional_synthesis(model, num_samples=args.n_samples, device=args.device)
    save_samples(x_hat, args.save_dir)
    if targets is not None:
        torch.save(targets, os.path.join(args.save_dir, "targets.pt"))
    if args.nearest_store is not None:
        from .data import PackedEmbeddingStore
        from .search import cosine_topk

        keys = PackedEmbeddingStore(args.nearest_store).to_device(args.device)[0]
        sim, idx = cosine_topk(x_hat.to(keys.device), keys, args.nearest_k)
        torch.save({"index": idx.cpu(), "similarity": sim.cpu()}, os.path.join(args.save_dir, "nearest.pt"))


if __name__ == "__main__":
    main()
