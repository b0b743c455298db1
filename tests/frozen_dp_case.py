"""One rank of the two-rank check of the classifier-only step (launched by torchrun from
tests/test_gpu_frozen_vae.py::test_frozen_vae_on_two_ranks).  Every rank prints one RESULT line: whether the ranks hold identical
parameters after frozen-VAE steps, whether the VAE stayed as it was, and how far they are from a single-process run on the whole batches."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist

    import pseudo_speaker_vae_b200 as P
    from pseudo_speaker_vae_b200 import _lib as L

    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    L.set_option("deterministic", 1)
    global_batch, calls = 2048, 5
    g = torch.Generator().manual_seed(13)
    xs = torch.randn(calls, global_batch, 256, generator=g)
    xs = xs / xs.norm(dim=2, keepdim=True)
    ys = torch.randint(0, 2, (calls, global_batch), generator=g)
    es = torch.randn(calls, global_batch, 64, generator=g)
    flats = {}
    for solo in (False, True):
        torch.manual_seed(3)
        m = P.PseudoSpeakerVAE(model=dict(input_dim=256, latent_dim=64), classifier=dict(input_dim=64, num_classes=2), optimizer=dict(lr=1e-3),
                               scheduler=dict(T_max=200), precision="bf16", freeze_vae=True).to(dev)
        start = m.hot_path.arena.flat.detach().clone()
        tr = P.DataParallelTrainer(m, local_only=solo)
        row0, rows = (0, global_batch) if solo else tr.set_shard(global_batch)
        m.hot_path.row0 = row0
        for s in range(calls):
            sl = slice(row0, row0 + rows)
            tr.train_step(xs[s, sl].to(dev), ys[s, sl].to(dev), es[s, sl].to(dev))
        torch.cuda.synchronize()
        a, _ = m.hot_path.classifier_span()
        flats[solo] = (m.hot_path.arena.flat.detach().double(), bool(torch.equal(m.hot_path.arena.flat[:a], start[:a])), tr.allreduce_kind)
    flat = flats[False][0].float()
    sig = torch.cat([flat.view(torch.int32).sum(dtype=torch.int64).reshape(1), flat.view(torch.int32)[::97].to(torch.int64)])
    sigs = [torch.empty_like(sig) for _ in range(dist.get_world_size())]
    dist.all_gather(sigs, sig)
    err = float((flats[False][0] - flats[True][0]).norm() / flats[True][0].norm())
    print("RESULT " + json.dumps(dict(rank=dist.get_rank(), ranks_identical=bool(all(torch.equal(s, sigs[0]) for s in sigs)), param_rel_err=err,
                                      vae_unchanged=flats[False][1] and flats[True][1], allreduce_kind=flats[False][2])), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
