#!/usr/bin/env python
"""Training step with loss_type='pde_loss': DeformerTrainer graph replay against the module path, device-timed.

    python scripts/pde_train_bench.py [--steps 30] [--warmup 10] [--rounds 3] [--only 2d_30x30 1d_200] [--out FILE.json]

Workloads (Poisson preset, mse(FEM solution, u_true_fine), Adam, lr 1e-3):
  2d_30x30   256 meshes of 30x30, Q = K = 101 (the shape of bench.py's f1 row: 101 x 101 evaluation grid);
  1d_200     4096 meshes of 200 nodes, Q = K = 101.
Module path: `model(data)` -> F.mse_loss(sol, u_true_fine) -> backward() -> torch.optim.Adam(fused=True).step().
Trainer: `step(sid)`, one CUDA-graph replay per step.  Each step is timed with CUDA events recorded on the stream it
runs on, before and after it, so launch gaps and host overhead that leave the device idle count.  The two paths
alternate in `rounds` blocks of `steps` steps each (after `warmup` steps of each), and the median per step over all
blocks is reported with the per-block medians.  The FEM forward and backward of the same batch are timed alone the same
way (library calls on the trainer slot's buffers).  The card name, power limit and max SM clock are printed with the
numbers.
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

from g_adaptivity_b200 import GNN, _lib, synth  # noqa: E402
from g_adaptivity_b200.trainer import DeformerTrainer  # noqa: E402

WORKLOADS = {
    "2d_30x30": ((30, 30), 256),
    "1d_200": ((200,), 4096),
}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    return q.stdout.strip()


def make(mesh_dims, B, dev):
    two_d = len(mesh_dims) == 2
    opt = synth.default_opt(mesh_dims, lr=1e-3, device=str(dev), gad_store_alpha=False, loss_type="pde_loss",
                            eval_quad_points=101, load_quad_points=101)
    ds = synth.SyntheticDataset(len(mesh_dims), mesh_dims, eval_quad_points=101 if two_d else None)
    data = synth.make_batch(mesh_dims, B, seed=0, eval_quad_points=101, with_u_true_fine=two_d)
    torch.manual_seed(42)
    state = copy.deepcopy(GNN(ds, opt).state_dict())
    return opt, ds, data, state


def timed(fn, stream, n):
    """Per-call device time (ms) of `n` calls of fn, events recorded on `stream` around each call."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for e0, e1 in ev:
        e0.record(stream)
        fn()
        e1.record(stream)
    stream.synchronize()
    return [e0.elapsed_time(e1) for e0, e1 in ev]


class ModulePath:
    def __init__(self, opt, ds, data, state, dev):
        self.model = GNN(ds, opt).to(dev)
        self.model.load_state_dict(state)
        self.model.train()
        self.optim = torch.optim.Adam(self.model.parameters(), lr=float(opt["lr"]), fused=True)
        self.d = data.to(dev)
        self.tgt = data.u_true_fine_tensor.to(dev)
        self.stream = torch.cuda.current_stream(dev)

    def step(self):
        self.optim.zero_grad(set_to_none=True)
        _, _, sol = self.model(self.d)
        self.loss = F.mse_loss(sol, self.tgt)
        self.loss.backward()
        self.optim.step()


class TrainerPath:
    def __init__(self, opt, ds, data, state, dev):
        self.model = GNN(ds, opt).to(dev)
        self.model.load_state_dict(state)
        self.tr = DeformerTrainer(self.model)
        self.sid = self.tr.add_batch(data)
        assert self.tr.slots[self.sid].pde
        self.stream = self.tr.stream

    def step(self):
        self.tr.step(self.sid)


def fem_calls(tr, s):
    """(forward, backward) of the slot's FEM stage alone, as library calls on the trainer's stream."""
    lib, P, chk, st = tr.lib, _lib.ptr, _lib.check, tr.stream.cuda_stream
    if tr.dim == 2:
        t, (ex, ey) = s.topo, s.eval_pts
        fem = (P(t.cells), t.T, P(t.is_bc), s.Nm, P(t.star_cell), P(t.star_loc), t.D, P(s.x_phys), P(s.centers),
               P(s.scales), s.G, s.B, s.K, P(ex), P(ey), s.Q)
        return (lambda: chk(lib.gad_fem2d_fwd(*fem, P(s.coeffs), P(s.sol), P(s.u64), P(s.cg_iters), st), "fwd"),
                lambda: chk(lib.gad_fem2d_bwd(*fem, P(s.u64), P(s.g_sol), P(s.g_out), st), "bwd"))
    fem = (P(s.x_phys), P(s.centers), P(s.scales), P(s.eval_pts[0]))
    return (lambda: chk(lib.gad_fem1d_fwd(*fem, s.B, s.Nm, s.G, s.K, s.Q, P(s.sol), None, st), "fwd"),
            lambda: chk(lib.gad_fem1d_bwd(*fem, P(s.g_sol), s.B, s.Nm, s.G, s.K, s.Q, P(s.g_out), st), "bwd"))


def med(xs):
    return round(statistics.median(xs), 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pde_train_bench.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    info = {"card": card(), "steps_per_block": a.steps, "warmup": a.warmup, "rounds": a.rounds}
    print(json.dumps(info), flush=True)
    rows = [info]
    for name in a.only:
        mesh_dims, B = WORKLOADS[name]
        opt, ds, data, state = make(mesh_dims, B, dev)
        paths = {"module": ModulePath(opt, ds, data, state, dev), "trainer": TrainerPath(opt, ds, data, state, dev)}
        for p in paths.values():
            timed(p.step, p.stream, a.warmup)
        samples = {k: [] for k in paths}
        blocks = {k: [] for k in paths}
        for _ in range(a.rounds):
            for k, p in paths.items():
                t = timed(p.step, p.stream, a.steps)
                samples[k] += t
                blocks[k].append(med(t))
        tr = paths["trainer"].tr
        fwd, bwd = fem_calls(tr, tr.slots[paths["trainer"].sid])
        timed(fwd, tr.stream, a.warmup)
        t_fwd = timed(fwd, tr.stream, a.steps)
        t_bwd = timed(bwd, tr.stream, a.steps)
        row = {"workload": name, "meshes": B, "nodes": int(data.x_comp.shape[0]), "Q": tr.slots[0].Q,
               "module_ms_per_step": med(samples["module"]), "trainer_ms_per_step": med(samples["trainer"]),
               "module_block_medians": blocks["module"], "trainer_block_medians": blocks["trainer"],
               "fem_fwd_ms": med(t_fwd), "fem_bwd_ms": med(t_bwd),
               "module_loss_last": float(paths["module"].loss.item()),
               "trainer_loss_last": float(tr.slots[0].loss.item())}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del paths, tr
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
