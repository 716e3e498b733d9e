#!/usr/bin/env python
"""Cost of global CNN features on meshes beyond one CTA: module forward + backward, device-timed, with and without
gnn_inc_glob_feat_f / _uu on the same model otherwise.

    python scripts/glob_large_bench.py [--iters 50] [--warmup 5] [--out FILE.json]

Workloads (L1 mesh loss, default model: hidden_dim 8, 4 layers, shared conv):
  16x64x64    16 meshes of 64x64,
  1x200x200   one 200x200 mesh,
each with ode_method euler and rk4, on the route the module's dispatch picks (cluster or streaming; reported per row).  Per workload the two models (with / without global features) run alternately in
the same process, `iters` calls each after `warmup` untimed calls: `model(data)` -> F.l1_loss -> backward(), between
CUDA events on a synchronised stream, gradients zeroed outside the timed window.  The model with global features also
runs its two CNNs (forward and backward) and the du product; that is part of what a user pays for the feature, and
is timed on its own as well (`us_cnn`: GNN._global_bias_offsets forward + backward of du.sum(), the same calls).
The card name, power limit and maximum SM clock are printed with the numbers (nvidia-smi).
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

WORKLOADS = {
    "16x64x64": ((64, 64), 16),
    "1x200x200": ((200, 200), 1),
}
GLOB = {"gnn_inc_glob_feat_f": True, "gnn_inc_glob_feat_uu": True}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    return q.stdout.strip()


def make_model(md, method, glob, dev):
    opt = synth.default_opt(md, device=str(dev), ode_method=method, gad_store_alpha=False, **(GLOB if glob else {}))
    ds = synth.SyntheticDataset(len(md), md)
    ds.x_comp_shared = synth.make_batch(md, 1).x_comp
    torch.manual_seed(42)
    model = GNN(ds, opt).to(dev)
    model.train()
    return model


def step(model, data, target):
    F.l1_loss(model(data), target).backward()


def cnn_step(model, data, dev):
    du = model._global_bias_offsets(data, model.last_graph, None, None, None, None, dev)
    du.sum().backward()


def timed(fn, model, iters):
    t = 0.0
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        t += e0.elapsed_time(e1)
        model.zero_grad(set_to_none=True)
    return 1000.0 * t / iters


def route(model):
    g = model.last_graph
    if g.tile_ptr is not None:
        return "mesh-resident"
    return "cluster" if getattr(g, "clf_in", None) is not None and g.cl_in is not None else "stream"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two models per workload")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("glob_large_bench.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    info = card()
    print(f"# {info}")
    rows = []
    for wname, (md, B) in WORKLOADS.items():
        data = synth.make_batch(md, B, seed=0)
        target = data.x_phys.to(dev)
        for method in ("euler", "rk4"):
            models = {g: make_model(md, method, g, dev) for g in (False, True)}
            for g, m in models.items():
                for _ in range(args.warmup):
                    step(m, data, target)
                    m.zero_grad(set_to_none=True)
            torch.cuda.synchronize()
            times = {False: [], True: [], "cnn": []}
            mg = models[True]
            for _ in range(args.rounds):
                for g, m in models.items():
                    times[g].append(timed(lambda: step(m, data, target), m, args.iters))
                times["cnn"].append(timed(lambda: cnn_step(mg, data, dev), mg, args.iters))
            base, glob = min(times[False]), min(times[True])
            row = dict(workload=wname, method=method, nodes=int(data.x_comp.shape[0]),
                       route_plain=route(models[False]), route_glob=route(models[True]),
                       us_plain=round(base, 1), us_glob=round(glob, 1), overhead=round(glob / base - 1.0, 4),
                       us_cnn=round(min(times["cnn"]), 1),
                       us_plain_rounds=[round(x, 1) for x in times[False]],
                       us_glob_rounds=[round(x, 1) for x in times[True]])
            rows.append(row)
            print(json.dumps(row), flush=True)
    out = {"card": info, "iters": args.iters, "rounds": args.rounds, "rows": rows}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
