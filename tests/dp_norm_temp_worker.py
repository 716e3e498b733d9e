"""Worker of tests/test_gpu_train_normalize_temperature.py: one rank of a data-parallel run with gnn_normalize=True
(torchrun, NCCL), alone and with a learnable temperature.  Every rank trains on its shard of the meshes of a global
batch; the shards' f / uu maxima differ, so each rank normalises by the MAX-all-reduced maxima of the union batch.
Rank 0 writes per configuration the parameters, whether the ranks agree, whether the shards' maxima differed and the
result of DeformerTrainer.dp_selfcheck."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch
import torch.distributed as dist


def _scale_features(data, B, first_mesh_id):
    # as tests/test_gpu_train_normalize_temperature.py:_scale_features
    n = data.f_tensor.numel() // B
    j = torch.arange(first_mesh_id, first_mesh_id + B, dtype=torch.float32).repeat_interleave(n)
    data.f_tensor = data.f_tensor * (1.0 + j % 3)
    data.uu_tensor = data.uu_tensor * (2.0 - 0.5 * (j % 2))
    return data


def main():
    out_path, steps, B = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from g_adaptivity_b200 import GNN, synth
    from g_adaptivity_b200.trainer import DeformerTrainer

    md = (12, 12)
    ds = synth.SyntheticDataset(2, md)
    res = {}
    for key, over in (("normalize", dict(gnn_normalize=True)),
                      ("normalize_learnable_a", dict(gnn_normalize=True, softmax_temp_type="learnable_a"))):
        opt = synth.default_opt(md, device=str(dev), gad_store_alpha=False, lr=1e-2, **over)
        torch.manual_seed(42)
        model = GNN(ds, opt).to(dev)
        tr = DeformerTrainer(model)
        batches = [_scale_features(synth.make_batch(md, B, seed=7, first_mesh_id=(k * world + rank) * B), B,
                                   (k * world + rank) * B) for k in range(2)]
        sids = [tr.add_batch(b) for b in batches]
        mine = torch.tensor([b.f_tensor.max().item() for b in batches], device=dev)
        every = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        for k in range(steps):
            tr.step(sids[k % 2])
        tr.synchronize()
        selfcheck = tr.dp_selfcheck(sids, steps=4)
        flat = tr.flat.detach().clone()
        gathered = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        res[key] = {"flat": flat.cpu().tolist(), "ranks_equal": all(bool(torch.equal(g, flat)) for g in gathered),
                    "shard_max_differ": not all(bool(torch.equal(e, every[0])) for e in every),
                    "peer_route": any(tr.slots[s].peer_route for s in sids), "selfcheck": selfcheck}
        tr.close()
    if rank == 0:
        with open(out_path, "w") as fh:
            json.dump(res, fh)
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    os._exit(0)      # skip NCCL teardown (graphs captured collectives): nothing left to clean up


if __name__ == "__main__":
    main()
