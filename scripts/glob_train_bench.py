#!/usr/bin/env python
"""Training step of a deformer with global CNN features: DeformerTrainer against the module path, device-timed.

    python scripts/glob_train_bench.py [--steps 100] [--warmup 10] [--out FILE.json]

Workloads (L1 mesh loss, Adam, lr 1e-3):
  2d_30x30   256 meshes of 30x30, gnn_inc_glob_feat_f (2-D CNN on the f grid of every mesh);
  1d_200     4096 meshes of 200 nodes (Burgers preset), gnn_inc_glob_feat_f and _uu (two 1-D CNNs).
Trainer: `run_epoch(timed=True)` over one captured graph of `steps` steps, `epoch_elapsed_ms` (device time between two
event-record nodes of that graph).  Module path: `model(data)` -> F.l1_loss -> backward() -> torch.optim.Adam(fused=True)
.step() with CUDA events around a synchronised loop of `steps` iterations.  Both start from the same parameters; after
the timed steps their parameters are compared (max |difference| / max |parameter|, lin_key.bias excluded: its gradient is
analytically zero).  The card name and power limit are printed with the numbers.
"""
import argparse
import copy
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from g_adaptivity_b200 import GNN, synth  # noqa: E402
from g_adaptivity_b200.trainer import DeformerTrainer  # noqa: E402

WORKLOADS = {
    "2d_30x30": ((30, 30), 256, False, {"gnn_inc_glob_feat_f": True}),
    "1d_200": ((200,), 4096, True, {"gnn_inc_glob_feat_f": True, "gnn_inc_glob_feat_uu": True}),
}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    return q.stdout.strip()


def make(mesh_dims, B, burgers, over, dev):
    opt = (synth.burgers_opt if burgers else synth.default_opt)(mesh_dims, lr=1e-3, device=str(dev),
                                                                gad_store_alpha=False, **over)
    ds = synth.SyntheticDataset(len(mesh_dims), mesh_dims)
    ds.x_comp_shared = synth.make_batch(mesh_dims, 1).x_comp
    data = synth.make_batch(mesh_dims, B, seed=0, burgers=burgers)
    torch.manual_seed(42)
    state = copy.deepcopy(GNN(ds, opt).state_dict())
    return opt, ds, data, state


def params(model):
    return {n: p.detach().cpu().clone() for n, p in model.named_parameters()}


def time_trainer(opt, ds, data, state, steps, warmup, dev):
    model = GNN(ds, opt).to(dev)
    model.load_state_dict(state)
    tr = DeformerTrainer(model, loss_fn="l1")
    sid = tr.add_batch(data)
    assert tr.slots[sid].glob
    tr.run_epoch([sid] * warmup, timed=True)
    tr.synchronize()
    tr.run_epoch([sid] * steps, timed=True)
    ms = tr.epoch_elapsed_ms([sid] * steps)
    tr.synchronize()
    return ms / steps, float(tr.slots[sid].loss.item()), params(model)


def time_module(opt, ds, data, state, steps, warmup, dev):
    model = GNN(ds, opt).to(dev)
    model.load_state_dict(state)
    model.train()
    optim = torch.optim.Adam(model.parameters(), lr=float(opt["lr"]), fused=True)
    d = data.to(dev)
    tgt = d.x_phys if d.x_phys.dim() == 2 else d.x_phys.unsqueeze(-1)

    def step():
        optim.zero_grad(set_to_none=True)
        loss = F.l1_loss(model(d), tgt)
        loss.backward()
        optim.step()
        return loss

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / steps, float(loss.item()), params(model)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--only", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("glob_train_bench.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    info = {"card": card(), "steps": a.steps, "warmup": a.warmup}
    print(json.dumps(info), flush=True)
    rows = [info]
    for name in a.only:
        mesh_dims, B, burgers, over = WORKLOADS[name]
        opt, ds, data, state = make(mesh_dims, B, burgers, over, dev)
        ms, loss, p_tr = time_trainer(opt, ds, data, state, a.steps, a.warmup, dev)
        ms_mod, loss_mod, p_mod = time_module(opt, ds, data, state, a.steps, a.warmup, dev)
        names = [n for n in p_mod if "lin_key.bias" not in n]
        scale = max(p_mod[n].abs().max().item() for n in names)
        dev_rel = max((p_tr[n] - p_mod[n]).abs().max().item() for n in names) / scale
        row = {"workload": name, "meshes": B, "nodes": int(data.x_comp.shape[0]),
               "trainer_us_per_step": round(ms * 1e3, 2), "module_us_per_step": round(ms_mod * 1e3, 2),
               "trainer_loss_last": loss, "module_loss_last": loss_mod,
               "params_max_rel_diff": dev_rel, "steps_compared": a.warmup + a.steps}
        print(json.dumps(row), flush=True)
        rows.append(row)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
