#!/usr/bin/env python
"""Training step with gnn_normalize=True or softmax_temp_type='learnable_a': DeformerTrainer graph replay against the
module path, device-timed.

    python scripts/normalize_temp_bench.py [--steps 50] [--warmup 10] [--rounds 3] [--only normalize learnable_a]
                                           [--out FILE.json]

Workload: 256 meshes of 30x30 (the shape of bench.py's cfg-2 row), mesh loss L1, Adam, lr 1e-3.
  normalize    module path and trainer with gnn_normalize=True, and the trainer on the same slot without it: the
               one-launch step with and without gad_batch_max in front (what the per-step maxima cost);
  learnable_a  module path and trainer with softmax_temp_type='learnable_a' (the trainer's chain of library kernels).
Module path: `model(data)` -> F.l1_loss -> backward() -> torch.optim.Adam(fused=True).step().  Trainer: `step(sid)`,
one CUDA-graph replay per step.  Each step is timed with CUDA events recorded on the stream it runs on, before and after
it, so launch gaps and host overhead that leave the device idle count.  The paths alternate in `rounds` blocks of
`steps` steps each (after `warmup` steps of each); the median per step over all blocks is reported with the per-block
medians.  The card name, power limit and max SM clock are printed with the numbers.
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from g_adaptivity_b200 import GNN, synth  # noqa: E402
from g_adaptivity_b200.trainer import DeformerTrainer  # noqa: E402

MESH, B = (30, 30), 256
WORKLOADS = {
    "normalize": dict(gnn_normalize=True),
    "learnable_a": dict(softmax_temp_type="learnable_a"),
}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    return q.stdout.strip()


def timed(fn, stream, n):
    """Per-call device time (ms) of `n` calls of fn, events recorded on `stream` around each call."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for e0, e1 in ev:
        e0.record(stream)
        fn()
        e1.record(stream)
    stream.synchronize()
    return [e0.elapsed_time(e1) for e0, e1 in ev]


def make_model(over, ds, state, dev):
    opt = synth.default_opt(MESH, lr=1e-3, device=str(dev), gad_store_alpha=False, **over)
    model = GNN(ds, opt).to(dev)
    model.load_state_dict(state)
    return model


class ModulePath:
    def __init__(self, model, data, dev):
        self.model = model
        self.model.train()
        self.optim = torch.optim.Adam(self.model.parameters(), lr=1e-3, fused=True)
        self.d = data.to(dev)
        self.tgt = data.x_phys.to(dev)
        self.stream = torch.cuda.current_stream(dev)

    def step(self):
        self.optim.zero_grad(set_to_none=True)
        out = self.model(self.d)
        self.loss = F.l1_loss(out, self.tgt)
        self.loss.backward()
        self.optim.step()


class TrainerPath:
    def __init__(self, model, data):
        self.tr = DeformerTrainer(model, loss_fn="l1")
        self.sid = self.tr.add_batch(data)
        self.stream = self.tr.stream
        s = self.tr.slots[self.sid]
        self.route = "chain" if s.chain else ("one-launch" if self.tr._one_launch(s) else "launch chain")
        self.loss = s.loss

    def step(self):
        self.tr.step(self.sid)


def med(xs):
    return round(statistics.median(xs), 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("normalize_temp_bench.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    info = {"card": card(), "meshes": B, "mesh": "x".join(map(str, MESH)), "steps_per_block": a.steps,
            "warmup": a.warmup, "rounds": a.rounds}
    print(json.dumps(info), flush=True)
    rows = [info]
    ds = synth.SyntheticDataset(2, MESH)
    data = synth.make_batch(MESH, B, seed=0)
    for name in a.only:
        over = WORKLOADS[name]
        torch.manual_seed(42)
        state = copy.deepcopy(GNN(ds, synth.default_opt(MESH, **over)).state_dict())
        paths = {"module": ModulePath(make_model(over, ds, state, dev), data, dev),
                 "trainer": TrainerPath(make_model(over, ds, state, dev), data)}
        if name == "normalize":      # the same slot without normalisation
            paths["trainer_plain"] = TrainerPath(make_model({}, ds, state, dev), data)
        for p in paths.values():
            timed(p.step, p.stream, a.warmup)
        samples = {k: [] for k in paths}
        blocks = {k: [] for k in paths}
        for _ in range(a.rounds):
            for k, p in paths.items():
                t = timed(p.step, p.stream, a.steps)
                samples[k] += t
                blocks[k].append(med(t))
        row = {"workload": name, "trainer_route": paths["trainer"].route}
        for k, p in paths.items():
            row[f"{k}_ms_per_step"] = med(samples[k])
            row[f"{k}_block_medians"] = blocks[k]
            row[f"{k}_loss_last"] = float(p.loss.item())
        print(json.dumps(row), flush=True)
        rows.append(row)
        del paths
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
