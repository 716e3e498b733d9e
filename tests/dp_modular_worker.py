"""Worker of tests/test_gpu_train_modular.py: one rank of a data-parallel run with loss_type='modular' (torchrun,
NCCL), on the in-kernel peer all-reduce and on NCCL.  Every rank trains on its shard of the meshes of a global batch
with the cotangent of its own shard: the outside loss is a mean over the union batch's nodes, so the shard's gradient
of its own mean is scaled by 1 / world, and the all-reduce sums the shards' gradients to the union batch's.  Rank 0
writes per route the parameters, whether the ranks agree, the route taken and DeformerTrainer.dp_selfcheck."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch
import torch.distributed as dist


def main():
    out_path, steps, B = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from g_adaptivity_b200 import GNN, synth
    from g_adaptivity_b200.trainer import DeformerTrainer
    from test_gpu_train_modular import _smooth_grad_fn

    md = (12, 12)
    ds = synth.SyntheticDataset(2, md)
    res = {}
    for key, over in (("peer", {}), ("nccl", {"gad_peer_allreduce": False})):
        opt = synth.default_opt(md, device=str(dev), gad_store_alpha=False, lr=1e-2, loss_type="modular", **over)
        torch.manual_seed(42)
        model = GNN(ds, opt).to(dev)
        tr = DeformerTrainer(model)
        batches = [synth.make_batch(md, B, seed=7, first_mesh_id=(k * world + rank) * B) for k in range(2)]
        sids = [tr.add_batch(b) for b in batches]
        for k in range(steps):
            b = batches[k % 2]
            x = tr.forward(sids[k % 2])
            tr.step(sids[k % 2], cotangent=_smooth_grad_fn(b.x_phys.to(dev))(x)[1] * (1.0 / world))
        tr.synchronize()
        selfcheck = tr.dp_selfcheck(sids, steps=4)
        flat = tr.flat.detach().clone()
        gathered = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        res[key] = {"flat": flat.cpu().tolist(), "ranks_equal": all(bool(torch.equal(g, flat)) for g in gathered),
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
