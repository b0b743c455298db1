"""One rank of the graphed data-parallel check (launched by torchrun from tests/test_gpu_graph.py::test_graphed_data_parallel_step_on_real_ranks,
or by hand: `python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/graph_dp_case.py`).  Every rank prints one RESULT
line: its graphed run (all-reduce inside the graph) against its eager run of the same steps, and whether the ranks hold identical parameters."""
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
    global_batch, steps = 4096, 6
    g = torch.Generator().manual_seed(11)
    xs = torch.randn(steps, global_batch, 256, generator=g)
    xs = xs / xs.norm(dim=2, keepdim=True)
    ys = torch.randint(0, 2, (steps, global_batch), generator=g)
    runs = {}
    for graphed in (False, True):
        torch.manual_seed(3)
        m = P.PseudoSpeakerVAE(model=dict(input_dim=256, latent_dim=64), classifier=dict(input_dim=64, num_classes=2), optimizer=dict(lr=1e-3),
                               scheduler=dict(T_max=200), precision="bf16").to(dev)
        m.hot_path.manual_seed(5, 0)
        tr = P.DataParallelTrainer(m)
        row0, rows = tr.set_shard(global_batch)
        step = P.GraphedTrainStep(tr, rows=rows) if graphed else tr.train_step
        for s in range(steps):
            step(xs[s, row0:row0 + rows].to(dev), ys[s, row0:row0 + rows].to(dev))
        torch.cuda.synchronize()
        runs[graphed] = (m.hot_path.arena.flat.detach().clone(), step if graphed else None)
    flat = runs[True][0]
    sig = torch.cat([flat.view(torch.int32).sum(dtype=torch.int64).reshape(1), flat.view(torch.int32)[::997].to(torch.int64)])
    sigs = [torch.empty_like(sig) for _ in range(dist.get_world_size())]
    dist.all_gather(sigs, sig)
    gs = runs[True][1]
    print("RESULT " + json.dumps(dict(rank=dist.get_rank(), bit_identical=bool(torch.equal(runs[True][0], runs[False][0])),
                                      ranks_identical=bool(all(torch.equal(s, sigs[0]) for s in sigs)), replays=gs.replays,
                                      allreduce_kind=gs.allreduce_kind, pdl=gs.pdl)), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
