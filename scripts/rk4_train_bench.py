#!/usr/bin/env python
"""Training step of an ode_method='rk4' deformer: DeformerTrainer against the module path, device-timed.

    python scripts/rk4_train_bench.py [--steps 200] [--warmup 20] [--out FILE.json]

Workloads (L = 4 RK4 steps, L1 mesh loss, Adam):
  cfg2_30x30   256 meshes of 30x30, the one-launch step (k_ell_train<..., GAD_METHOD_RK4>);
  1d_200       4096 meshes of 200 nodes, the one-launch step (CE = 2);
  chain_50x50  1024 meshes of 50x50, the launch chain (tiles too large for the one-launch kernel's rows).
Trainer: `run_epoch(timed=True)` over one graph of `steps` PDL-chained steps, `epoch_elapsed_ms` (device time between
two event-record nodes of that graph).  Module path: `model(data)` -> F.l1_loss -> backward() -> torch.optim.Adam.step()
with CUDA events around a synchronised loop of `steps` iterations.

Roofline: the streaming byte model of DESIGN §4 counted for RK4 -- per node and step, 7 forward F-evaluations (4, plus
3 recomputed in the backward) of 8·C + 4·d + 4 bytes and 4 vjp pass pairs of 12·C + 2·(4·d + 4) bytes, plus the
inputs 4·in_dim + 8·dim once (C live channels, d = E / N).  The fraction is against the device-to-device copy rate
measured in the same run (and the data sheet's 7.7 TB/s, for reference).  The card name and power limit are printed
with the numbers.
"""
import argparse
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
    "cfg2_30x30": ((30, 30), 256, False),
    "1d_200": ((200,), 4096, True),
    "chain_50x50": ((50, 50), 1024, False),
}
DATASHEET_BW = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    return q.stdout.strip()


def copy_rate(dev):
    """Device-to-device copy of 2 GiB (far beyond the 126 MB L2): bytes read + written per second."""
    n = 1 << 29
    a = torch.empty(n, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    e1.synchronize()
    return 10 * 2 * a.numel() * 4 / (e0.elapsed_time(e1) * 1e-3)


def make(mesh_dims, B, burgers, dev):
    opt = (synth.burgers_opt if burgers else synth.default_opt)(mesh_dims, ode_method="rk4", num_layers=4, lr=1e-3,
                                                                device=str(dev), gad_store_alpha=False)
    ds = synth.SyntheticDataset(len(mesh_dims), mesh_dims)
    data = synth.make_batch(mesh_dims, B, seed=0, burgers=burgers)
    torch.manual_seed(42)
    return opt, ds, data


def bytes_per_node(model, graph, in_dim):
    C, L, dim = model.CE, int(model.opt["num_layers"]), model.dim
    d = graph.E / graph.N
    bf, bb = 8 * C + 4 * d + 4, 12 * C + 2 * (4 * d + 4)
    return L * (7 * bf + 4 * bb) + 4 * in_dim + 8 * dim


def time_trainer(opt, ds, data, steps, warmup, dev):
    model = GNN(ds, opt).to(dev)
    tr = DeformerTrainer(model, loss_fn="l1")
    sid = tr.add_batch(data)
    one_launch = tr._one_launch(tr.slots[sid])
    tr.run_epoch([sid] * warmup, timed=True)
    tr.synchronize()
    tr.run_epoch([sid] * steps, timed=True)
    ms = tr.epoch_elapsed_ms([sid] * steps)
    tr.synchronize()
    loss = float(tr.slots[sid].loss.item())
    g = tr.slots[sid].graph
    in_dim = model.dim + int(bool(opt["gnn_inc_feat_f"])) + int(bool(opt["gnn_inc_feat_uu"]))
    return ms / steps, one_launch, loss, bytes_per_node(model, g, in_dim), g.N


def time_module(opt, ds, data, steps, warmup, dev):
    model = GNN(ds, opt).to(dev)
    model.train()
    optim = torch.optim.Adam(model.parameters(), lr=float(opt["lr"]))
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
    return e0.elapsed_time(e1) / steps, float(loss.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--only", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rk4_train_bench.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    info = {"card": card(), "copy_rate_GBps": round(copy_rate(dev) / 1e9, 1), "steps": a.steps, "warmup": a.warmup}
    print(json.dumps(info), flush=True)
    rows = [info]
    for name in a.only:
        mesh_dims, B, burgers = WORKLOADS[name]
        opt, ds, data = make(mesh_dims, B, burgers, dev)
        ms, one_launch, loss, bpn, N = time_trainer(opt, ds, data, a.steps, a.warmup, dev)
        ms_mod, loss_mod = time_module(opt, ds, data, a.steps, a.warmup, dev)
        alg = bpn * N / (ms * 1e-3)
        row = {"workload": name, "meshes": B, "nodes": N, "route": "one launch" if one_launch else "launch chain",
               "trainer_us_per_step": round(ms * 1e3, 2), "module_us_per_step": round(ms_mod * 1e3, 2),
               "speedup": round(ms_mod / ms, 2), "trainer_mesh_nodes_per_s": round(N / (ms * 1e-3) / 1e9, 3),
               "module_mesh_nodes_per_s": round(N / (ms_mod * 1e-3) / 1e9, 3), "nodes_per_s_unit": "G",
               "algorithmic_bytes_per_node": round(bpn, 1),
               "roofline_fraction_of_copy_rate": round(alg / (info["copy_rate_GBps"] * 1e9), 3),
               "roofline_fraction_of_datasheet": round(alg / DATASHEET_BW, 3),
               "trainer_loss_last": loss, "module_loss_last": loss_mod}
        print(json.dumps(row), flush=True)
        rows.append(row)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
