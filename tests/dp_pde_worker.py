"""Worker of tests/test_gpu_train_pde_loss.py: one rank of a data-parallel run with loss_type='pde_loss' (torchrun,
NCCL).  Every rank trains on its shard of the meshes of a global batch; rank 0 writes the parameters, whether the ranks
agree, the slot's route and the result of DeformerTrainer.dp_selfcheck."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

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

    md, Q = (7, 7), 13
    ds = synth.SyntheticDataset(2, md, eval_quad_points=Q)
    opt = synth.default_opt(md, device=str(dev), gad_store_alpha=False, lr=1e-2, eval_quad_points=Q, load_quad_points=9,
                            loss_type="pde_loss")
    torch.manual_seed(42)
    model = GNN(ds, opt).to(dev)
    tr = DeformerTrainer(model)
    sids = [tr.add_batch(synth.make_batch(md, B, seed=7, first_mesh_id=(k * world + rank) * B, eval_quad_points=Q,
                                          with_u_true_fine=True)) for k in range(2)]
    for k in range(steps):
        tr.step(sids[k % 2])
    tr.synchronize()
    selfcheck = tr.dp_selfcheck(sids, steps=4)
    flat = tr.flat.detach().clone()
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    res = {"flat": flat.cpu().tolist(), "ranks_equal": all(bool(torch.equal(g, flat)) for g in gathered),
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
