#!/usr/bin/env python
"""Training step with loss_type='modular' (the caller computes the cotangent of x_phys): DeformerTrainer against the
module loop, device-timed.

    python scripts/modular_train_bench.py [--steps 50] [--warmup 10] [--rounds 3] [--only cfg2 burgers] [--out FILE.json]

Workloads: `cfg2`, 256 meshes of 30x30 (the shape of bench.py's cfg-2 row); `burgers`, the reference's Burgers preset
(synth.burgers_opt: GRAND conv, 1-D meshes of 21 nodes) at 4096 meshes.  Adam, lr 1e-3.  The outside gradient is the
same torch expression on the device in both paths, g = tanh(x - target) / count.
  module   `out = model(data)` -> g(out.detach()) -> `(out * g).sum().backward()` -> torch.optim.Adam(fused=True).step();
  trainer  `x = trainer.forward(sid)` -> g(x) -> `trainer.step(sid, cotangent=g)`, each a CUDA-graph replay; the step
           recomputes its forward, so its one-launch route stays one launch.
Also timed alone on the trainer: `forward` (the recomputed forward's share of an iteration) and `step` with a resident
cotangent.  Each iteration is timed with CUDA events on the caller's stream (which waits for the trainer stream before
the closing record), so launch gaps and host overhead that leave the device idle count.  The paths alternate in `rounds`
blocks of `steps` iterations (after `warmup` of each); the median per iteration over all blocks is reported with the
per-block medians.  The card name, power limit and max SM clock are read in the same run and printed with the numbers.
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

from g_adaptivity_b200 import GNN, synth  # noqa: E402
from g_adaptivity_b200.trainer import DeformerTrainer  # noqa: E402

WORKLOADS = {
    "cfg2": dict(mesh=(30, 30), B=256, burgers=False),
    "burgers": dict(mesh=(21,), B=4096, burgers=True),
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


def outside_grad(x, target):
    return torch.tanh(x - target) * (1.0 / x.numel())


def make_opt(w, dev):
    mk = synth.burgers_opt if w["burgers"] else synth.default_opt
    return mk(w["mesh"], lr=1e-3, device=str(dev), gad_store_alpha=False, loss_type="modular")


class ModulePath:
    def __init__(self, model, data, dev):
        self.model = model
        self.model.train()
        self.optim = torch.optim.Adam(self.model.parameters(), lr=1e-3, fused=True)
        self.d = data.to(dev)
        self.tgt = None

    def step(self):
        self.optim.zero_grad(set_to_none=True)
        out = self.model(self.d)
        if self.tgt is None:
            self.tgt = self.d.x_phys.reshape(out.shape)
        (out * outside_grad(out.detach(), self.tgt)).sum().backward()
        self.optim.step()


class TrainerPath:
    def __init__(self, model, data, dev):
        self.tr = DeformerTrainer(model)
        self.sid = self.tr.add_batch(data)
        s = self.tr.slots[self.sid]
        self.route = "chain" if s.chain else ("one-launch" if self.tr._one_launch(s) else "launch chain")
        self.tgt = data.x_phys.to(dev).reshape(s.x_phys.shape)
        self.cur = torch.cuda.current_stream(dev)
        self.g = torch.zeros_like(s.x_phys)

    def step(self):
        x = self.tr.forward(self.sid)
        self.tr.step(self.sid, cotangent=outside_grad(x, self.tgt))
        self.cur.wait_stream(self.tr.stream)

    def forward_only(self):
        self.tr.forward(self.sid)

    def step_only(self):
        self.tr.step(self.sid, cotangent=self.g)
        self.cur.wait_stream(self.tr.stream)


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
        raise SystemExit("modular_train_bench.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    info = {"card": card(), "steps_per_block": a.steps, "warmup": a.warmup, "rounds": a.rounds}
    print(json.dumps(info), flush=True)
    rows = [info]
    for name in a.only:
        w = WORKLOADS[name]
        ds = synth.SyntheticDataset(len(w["mesh"]), w["mesh"])
        data = synth.make_batch(w["mesh"], w["B"], seed=0, burgers=w["burgers"])
        opt = make_opt(w, dev)
        torch.manual_seed(42)
        state = copy.deepcopy(GNN(ds, opt).to(dev).state_dict())
        models = [GNN(ds, opt).to(dev) for _ in range(2)]
        for m in models:
            m.load_state_dict(state)
        tp = TrainerPath(models[1], data, dev)
        cur = torch.cuda.current_stream(dev)
        paths = {"module": ModulePath(models[0], data, dev).step, "trainer": tp.step,
                 "trainer_forward": tp.forward_only, "trainer_step": tp.step_only}
        for fn in paths.values():
            timed(fn, cur, a.warmup)
        samples = {k: [] for k in paths}
        blocks = {k: [] for k in paths}
        for _ in range(a.rounds):
            for k, fn in paths.items():
                t = timed(fn, cur, a.steps)
                samples[k] += t
                blocks[k].append(med(t))
        row = {"workload": name, "meshes": w["B"], "mesh": "x".join(map(str, w["mesh"])), "trainer_route": tp.route}
        for k in paths:
            row[f"{k}_ms"] = med(samples[k])
            row[f"{k}_block_medians"] = blocks[k]
        row["speedup_module_over_trainer"] = round(row["module_ms"] / row["trainer_ms"], 2)
        row["forward_share_of_step"] = round(row["trainer_forward_ms"] / row["trainer_step_ms"], 3)
        print(json.dumps(row), flush=True)
        rows.append(row)
        del paths, tp, models
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
