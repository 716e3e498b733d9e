#!/usr/bin/env python
"""Headline benchmark: mesh-nodes/s through the deformer forward+backward (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): batched 2D 30x30 meshes, batch 256 per GPU, 4 Euler layers,
hidden 8, fp32, L1 mesh loss -- one STEP is one full training pass over one batch: feature
assembly -> L Euler layers -> loss/cotangent -> backward -> weight gradients -> [NCCL gradient
all-reduce when N > 1] -> Adam -> refold of the projection.  On one GPU that is ONE kernel launch
(`gad_train_step_ell`, csrc/ell_kernels.cuh: k_ell_train); with N > 1 ranks the kernel stops after
the weight gradients and all-reduce, Adam and the refold follow.  Weak scaling: every rank owns
its own 256-mesh shard (no data-path collective, SURVEY 8e).

L2 hygiene: the timed loop walks a ring of R distinct resident batches (own features, own graph
arrays) whose read-only footprint exceeds the 126 MB L2 several times over, so no step finds
its inputs in L2 ("config.l2").

Printed JSON (rank 0, one line): `value` = nodes/s with inputs resident in HBM (CUDA-graph
replay, device-timed, max over ranks); `e2e` = the same step driven from pinned HOST buffers
through `DeformerTrainer.run_from_host` (every step: H2D of its features/targets on a copy stream,
D2H of its loss; both inside the timed region); `roofline` = algorithmic bytes of the dominant
kernel (the one-launch train kernel) / its CUDA-event duration against the measured HBM peak; `cpu_baseline` = the CPU oracle (port of the
reference path) timed on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

MESH_DIMS = (30, 30)
MESHES_PER_GPU = 256
NUM_LAYERS = 4
METRIC = "mesh_nodes_per_sec_deformer_fwd_bwd"
UNIT = "nodes/s"
# the same string on both arms (the driver compares the arms' `config.workload`)
WORKLOAD = (f"cfg2: {MESHES_PER_GPU} x {MESH_DIMS[0]}x{MESH_DIMS[1]} meshes per GPU, fwd+bwd train step "
            f"(L={NUM_LAYERS} Euler layers, hidden 8, L1 mesh loss, Adam)")
GRAPH_STEPS = 256       # most training steps held by one CUDA graph of the timed region


# ------------------------------------------------------------------------------------------
# algorithmic bytes (SURVEY 8d): per node per F-evaluation, fp32 state, int32 indices
# ------------------------------------------------------------------------------------------
def algorithmic_bytes(n_nodes: int, n_edges: int, c_eff: int, L: int, in_dim: int, dim: int):
    dbar = n_edges / n_nodes
    b_f = 8 * c_eff + 4 * dbar + 4
    b_b = 12 * c_eff + 2 * (4 * dbar + 4)
    fwd = L * b_f + 4 * in_dim + 4 * dim
    bwd = L * b_b + 4 * dim
    return {"dbar": dbar, "fwd_per_node": fwd, "bwd_per_node": bwd, "step_per_node": fwd + bwd}


def ncu_traffic(kernel: str):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/traffic.json,
    written by scripts/ncu_traffic.py from an `ncu --set full` report of this command), or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as fh:
        return json.load(fh).get(kernel, {}).get("dram_bytes_per_launch")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
# clocks (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self, start: bool):
        if start:
            self.t0 = time.time()
        else:
            self.t1 = time.time()

    def stop(self):
        if self.proc is not None:
            # reap the sampler: bench.py must not leave an nvidia-smi process (or its zombie) behind
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
                self.proc.wait()
        sm, smax, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        lo = (self.t0 or 0) - 0.05
        hi = (self.t1 or time.time()) + 0.05
        rows = [r for t, r in self.rows if lo <= t <= hi] or [r for _, r in self.rows]
        for r in rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU oracle timing (cpu_baseline and --impl reference)
# ------------------------------------------------------------------------------------------
def time_cpu_oracle(steps: int, warmup: int, budget_s: float = 25.0, meshes: int = MESHES_PER_GPU):
    """One training step of the CPU oracle (pure-PyTorch port of the reference path; PyG itself is not
    installable here): forward + L1 mesh loss + autograd backward + torch.optim.Adam step
    (src/run_GNN.py:88,99-131) on a batch of `meshes` 30x30 meshes, all host threads."""
    import copy
    from g_adaptivity_b200 import synth
    from oracle import gnn_oracle

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    opt = synth.default_opt(MESH_DIMS, num_layers=NUM_LAYERS)
    ds = synth.SyntheticDataset(2, MESH_DIMS)
    data = synth.make_batch(MESH_DIMS, meshes, seed=0)
    torch.manual_seed(42)
    model = gnn_oracle.GNNRef(ds, copy.deepcopy(opt))
    model.train()
    optim = torch.optim.Adam(model.parameters(), lr=opt["lr"], weight_decay=opt["decay"])
    n_nodes = data.x_comp.shape[0]

    def one():
        optim.zero_grad(set_to_none=True)
        out = model(data)
        gnn_oracle.mesh_loss(out, data.x_phys).backward()
        optim.step()

    for _ in range(max(1, warmup)):
        one()
    times = []
    t_start = time.perf_counter()
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    ms = 1e3 * sum(times) / len(times)
    return {"value": n_nodes / (ms * 1e-3), "ms_per_step": ms, "cores": cores, "steps": len(times),
            "sample": f"{meshes} meshes of {MESH_DIMS[0]}x{MESH_DIMS[1]} ({n_nodes} nodes) per step, "
                      f"fwd + L1 loss + autograd bwd + torch.optim.Adam, torch CPU {torch.get_num_threads()} threads, "
                      f"mean of {len(times)} steps"}


def run_reference(args, rank: int, world: int):
    """Reference arm: the reference's CPU implementation of the path.  The reference itself cannot
    run here (torch_geometric / Firedrake absent, SURVEY 8c), so this times the oracle port: exactly
    `--warmup` + `--steps` steps of the same workload; when that many full batches would take more than a
    few minutes the step becomes a bounded sample (fewer meshes of the same shape per step)."""
    if rank != 0:
        return
    W, K = max(3, args.warmup), max(1, args.steps)
    meshes = MESHES_PER_GPU
    while meshes > 1 and (W + K) * 1.2 * meshes / MESHES_PER_GPU > 150.0:    # ~1.2 s per full batch on 16 cores
        meshes //= 2
    r = time_cpu_oracle(K, W, budget_s=240.0, meshes=meshes)
    n_nodes = MESHES_PER_GPU * MESH_DIMS[0] * MESH_DIMS[1]
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": W, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "nodes_per_step_per_gpu": n_nodes, "device": "host CPU",
                   "meshes_per_cpu_step": meshes},
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# the other BASELINE.json configs under the same clock (device-timed; reported in `configs`, not as `value`)
# ------------------------------------------------------------------------------------------
def fwd_bytes_per_node(N, E, ce, fevals, in_dim, dim):
    return fevals * (8 * ce + 4 * E / N + 4) + 4 * in_dim + 4 * dim


def time_forward_config(dev, md, B, over, burgers, iters, peak):
    """Forward through the module seam (`model(data)` under no_grad, inputs device-resident) and through
    `model.inference_session(data)` (one CUDA-graph replay per call, new `uu` copied in each time)."""
    from g_adaptivity_b200 import GNN, synth
    opt = synth.burgers_opt(md) if burgers else synth.default_opt(md)
    opt.update(device=str(dev), gad_store_alpha=False, gad_sync_timestamp=False, **over)     # throughput: no per-call sync
    ds = synth.SyntheticDataset(len(md), md)
    torch.manual_seed(42)
    model = GNN(ds, opt).to(dev).eval()
    data = synth.make_batch(md, B, seed=0, burgers=burgers).to(dev)
    with torch.no_grad():
        for _ in range(3):
            model(data)
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            model(data)
            e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        sess = model.inference_session(data)
        for _ in range(3):
            sess()
        torch.cuda.synchronize(dev)
        n_rep = max(20, iters)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_rep):
            sess(uu=data.uu_tensor)
        e1.record()
        torch.cuda.synchronize(dev)
        ms_sess = e0.elapsed_time(e1) / n_rep
        # the same replay as the device sees it: the host queues all replays behind a spin, CUDA-event pairs on the
        # session's stream time each one (graph launch on the device + kernels, no host call in between)
        pairs = []
        with torch.cuda.stream(sess.stream):
            torch.cuda._sleep(int(4e7))
            for _ in range(n_rep):
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record(sess.stream)
                sess.cuda_graph.replay()
                a1.record(sess.stream)
                pairs.append((a0, a1))
        sess.stream.synchronize()
        ms_dev = statistics.median(a0.elapsed_time(a1) for a0, a1 in pairs[2:])
    g = model.last_graph
    ms = statistics.median(ts)
    fevals = opt["num_layers"] * (4 if opt.get("ode_method", "euler") == "rk4" else 1)
    bpn = fwd_bytes_per_node(g.N, g.E, model.live, fevals, sum(model.in_dims), model.dim)
    return {"nodes": g.N, "edges": g.E, "f_evaluations": fevals, "bytes_per_node": round(bpn, 1),
            "module_call": {"ms": round(ms, 4), "nodes_per_s": g.N / (ms * 1e-3),
                            "roofline_frac": g.N * bpn / (ms * 1e-3) / 1e9 / peak},
            "device_replay": {"ms": round(ms_dev, 4), "nodes_per_s": g.N / (ms_dev * 1e-3),
                              "roofline_frac": g.N * bpn / (ms_dev * 1e-3) / 1e9 / peak,
                              "what": "the session's graph replayed back to back, CUDA events around each replay "
                                      "(no host call between replays; the call's inputs stay in L2 between replays, as they do between "
                                      "the repeated calls of a rollout)"},
            "session_replay": {"ms": round(ms_sess, 4), "nodes_per_s": g.N / (ms_sess * 1e-3),
                               "roofline_frac": g.N * bpn / (ms_sess * 1e-3) / 1e9 / peak}}


def time_cfg5(dev, rank, world, iters, peak, barrier):
    """BASELINE configs[4]: data-parallel training on 50x50 meshes, GLOBAL batch 8192 (strong scaling: 8192 / N
    meshes per GPU), one optimizer step per global batch, gradient all-reduce inside the kernel."""
    import torch.distributed as dist
    from g_adaptivity_b200 import GNN, synth
    from g_adaptivity_b200.trainer import DeformerTrainer
    md, total = (50, 50), 8192
    per = total // world
    opt = synth.default_opt(md, device=str(dev), gad_store_alpha=False, gad_shared_topology=True)
    ds = synth.SyntheticDataset(2, md)
    torch.manual_seed(42)
    model = GNN(ds, opt).to(dev)
    tr = DeformerTrainer(model)
    tr.broadcast_parameters()
    ring = 2
    sids = [tr.add_batch(synth.make_batch_device(md, per, dev, seed=500 + 7 * r + 1000 * rank)) for r in range(ring)]
    key = tuple(sids) * 2
    tr.capture_epoch(key)
    tr.run_epoch(key)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(tr.stream)
    for _ in range(iters):
        tr.run_epoch(key)
    e1.record(tr.stream)
    barrier()
    tr.check_peer()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / (iters * len(key))
    s0 = tr.slots[0]
    N, E = s0.N, s0.graph.E
    ab = algorithmic_bytes(N, E, model.live, opt["num_layers"], sum(model.in_dims), model.dim)
    out = {"workload": f"cfg5: global batch {total} x 50x50 meshes, {per} per GPU (strong scaling), train step",
           "nodes_per_gpu": N, "ms_per_step": round(ms, 4), "nodes_per_s": world * N / (ms * 1e-3),
           "bytes_per_node": round(ab["step_per_node"], 1),
           "roofline_frac": N * ab["step_per_node"] / (ms * 1e-3) / 1e9 / peak,
           "data": "256 distinct samples per GPU tiled on the device (synth.make_batch_device)",
           "topology": "shared (one ELL table)" if s0.graph.uniform else "general",
           "one_launch": bool(tr._one_launch(s0))}
    tr.close()
    del tr, model
    torch.cuda.empty_cache()
    return out


def time_pde_loss_2d(dev, iters):
    """Row f1: the reference's DEFAULT loss (`loss_type='pde_loss'`, params.py:109) on cfg-2-shaped data through the
    module seam: model(data) = deformer + batched 2-D FEM solve (csrc/fem2d.cu; the reference loops torch_FEM_2D per
    mesh in Python, src/GNN.py:327-335) -> mse(sol, u_true_fine) -> backward -> torch.optim.Adam; inputs resident."""
    import torch.nn.functional as F
    from g_adaptivity_b200 import GNN, synth
    md, B, Q = MESH_DIMS, MESHES_PER_GPU, 101
    opt = synth.default_opt(md, device=str(dev), gad_store_alpha=False, loss_type="pde_loss", eval_quad_points=Q,
                            load_quad_points=101)
    ds = synth.SyntheticDataset(2, md, eval_quad_points=Q)
    torch.manual_seed(42)
    model = GNN(ds, opt).to(dev).train()
    optim = torch.optim.Adam(model.parameters(), lr=1e-3)
    data = synth.make_batch(md, B, seed=0, eval_quad_points=Q, with_u_true_fine=True).to(dev)
    tgt = data.u_true_fine_tensor
    ts, fem = [], []
    for it in range(iters + 2):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        optim.zero_grad(set_to_none=True)
        e0.record()
        coeffs, xp, sol = model(data)
        loss = F.mse_loss(sol, tgt)
        loss.backward()
        e1.record()
        optim.step()
        e2.record()
        torch.cuda.synchronize(dev)
        if it >= 2:
            ts.append(e0.elapsed_time(e2))
    ms = statistics.median(ts)
    return {"workload": f"{B} x {md[0]}x{md[1]} meshes, loss_type='pde_loss' (deformer + batched 2-D FEM solve, 101-point "
                        "load cubature, 101x101 evaluation grid), fwd + bwd + torch Adam through GNN.forward",
            "ms_per_step": round(ms, 3), "meshes_per_s": B / (ms * 1e-3), "loss": float(loss.item()),
            "reference": "torch_FEM_2D per mesh in a Python loop: ~3 s per 30x30 mesh on the CPU (DESIGN section 11)"}


def time_loop_shape(dev, iters):
    """cfg 2 in the REFERENCE's loop shape (src/run_GNN.py:97-131): a fresh pinned host Batch per iteration.
    (a) the module seam exactly as the reference writes it: model(data) -> F.l1_loss -> backward() ->
    torch.optim.Adam.step(); (b) the same loop body as ONE call, `DeformerTrainer.train_batch(data)` (H2D of the
    batch's node inputs on a copy stream + the one-launch training step).  Wall clock per iteration, pipelined."""
    import torch.nn.functional as F
    from g_adaptivity_b200 import GNN, synth
    from g_adaptivity_b200.trainer import DeformerTrainer
    md, B = MESH_DIMS, MESHES_PER_GPU
    opt = synth.default_opt(md, device=str(dev), gad_store_alpha=False, gad_shared_topology=True)
    ds = synth.SyntheticDataset(2, md)
    base = synth.make_batch(md, B, seed=0)
    batches = []
    for _ in range(iters + 6):
        b = base.clone()
        b.pin_memory()
        batches.append(b)
    out = {}
    torch.manual_seed(42)
    model = GNN(ds, dict(opt)).to(dev).train()
    optim = torch.optim.Adam(model.parameters(), lr=1e-3, fused=True)
    for k, d in enumerate(batches):
        if k == 6:
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
        optim.zero_grad(set_to_none=True)
        F.l1_loss(model(d), d.x_phys.to(dev, non_blocking=True)).backward()
        optim.step()
    torch.cuda.synchronize(dev)
    out["module_seam_ms"] = round(1e3 * (time.perf_counter() - t0) / iters, 4)
    torch.manual_seed(42)
    model2 = GNN(ds, dict(opt)).to(dev).train()
    tr = DeformerTrainer(model2)
    for k, d in enumerate(batches):
        if k == 6:
            tr.synchronize()
            t0 = time.perf_counter()
        loss = tr.train_batch(d)
    tr.synchronize()
    ms = 1e3 * (time.perf_counter() - t0) / iters
    out["train_batch_ms"] = round(ms, 4)
    out["train_batch_nodes_per_s"] = B * md[0] * md[1] / (ms * 1e-3)
    out["workload"] = (f"{B} x {md[0]}x{md[1]} meshes, a fresh pinned host Batch per iteration: model(data) + F.l1_loss + "
                       "backward + torch.optim.Adam(fused) vs DeformerTrainer.train_batch(data)")
    tr.close()
    return out


def bind_rank_to_cores(local_rank: int, local_world: int):
    """One process per GPU on a shared host: give every rank its own slice of the cores this job may use, so
    that the ranks' launch / copy threads do not migrate over each other (all GPUs of the box report the same
    CPU affinity, `nvidia-smi topo -m`).  Memory is first-touched (and pinned) by the bound thread afterwards.
    Returns the core list, or None where the platform has no sched_setaffinity."""
    if local_world <= 1 or not hasattr(os, "sched_setaffinity"):
        return None
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // local_world
        if per < 1:
            return None
        mine = cores[local_rank * per:(local_rank + 1) * per]
        os.sched_setaffinity(0, mine)
        torch.set_num_threads(max(1, min(per, 4)))
        return [mine[0], mine[-1]]
    except OSError:
        return None


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ring", type=int, default=32, help="distinct resident batches walked by the timed loop")
    ap.add_argument("--no-shared-topology", action="store_true", help="build the general graph of the whole batch")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-epoch", action="store_true", help="one CUDA graph per step instead of one per pass over the ring")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--write-combined", action="store_true", help="e2e: packed host batches in write-combined pinned memory")
    ap.add_argument("--relay", default="auto", choices=["auto", "off"],
                    help="e2e at N > 1: balance unequal host->device paths by relaying part of some ranks' batches "
                         "through other ranks' GPUs (NVLink); proposals are timed on the real loop and the direct loop "
                         "stays unless one of them is at least 3%% faster (DESIGN section 15)")
    ap.add_argument("--skip-configs", action="store_true", help="do not time the other BASELINE configs (cfg 1, 3, 4, 5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy: loss, x_phys (the deformed "
                         "mesh of its batch), params and grads (the flat parameter vector after its Adam update and the "
                         "gradient it applied); inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the CUDA training step (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from g_adaptivity_b200 import GNN, _lib, synth
    from g_adaptivity_b200.trainer import DeformerTrainer

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the deformer has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity = bind_rank_to_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)
    K = max(1, args.steps)
    R = max(1, args.ring)

    # ---- workload ----------------------------------------------------------------------
    # the synthetic dataset is on one shared mesh, as the reference's `randg` datasets (src/data.py:143): the
    # graph is built for one tile and every tile of the batch uses that ELL table (row f2, MeshGraph.build_uniform)
    opt = synth.default_opt(MESH_DIMS, num_layers=NUM_LAYERS, device=str(dev), gad_store_alpha=False,
                            gad_shared_topology=not args.no_shared_topology)
    ds = synth.SyntheticDataset(2, MESH_DIMS)
    torch.manual_seed(42)
    model = GNN(ds, opt).to(dev)
    trainer = DeformerTrainer(model, use_cuda_graph=not args.no_graph)
    trainer.broadcast_parameters()
    host_batches = []
    for r in range(R):
        first = (rank * R + r) * MESHES_PER_GPU
        b = synth.make_batch(MESH_DIMS, MESHES_PER_GPU, seed=1000, first_mesh_id=first)
        b.pin_memory()
        host_batches.append(b)
        trainer.add_batch(b)
    s0 = trainer.slots[0]
    n_nodes, n_edges = s0.N, s0.graph.E
    in_dim = sum(model.in_dims)
    ab = algorithmic_bytes(n_nodes, n_edges, model.live, NUM_LAYERS, in_dim, model.dim)
    per_slot = lambda s: [s.inbuf] + ([] if s.graph.uniform else [s.graph.ell_in, s.graph.ell_out])
    ro_bytes = sum(t.numel() * t.element_size() for s in trainer.slots for t in per_slot(s))
    lib = _lib.load()

    if not args.no_graph:
        for sid in range(R):
            trainer.capture(sid)
    trainer.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()

    # ---- device-resident timing: >= W warm-up steps + exactly K timed steps -----------------
    # The K timed steps are CUDA-graph replays: one graph holds up to GRAPH_STEPS consecutive steps over
    # the ring of resident batches (consecutive steps linked by programmatic dependent launch); K steps =
    # n_full replays of the G-step graph + one replay of a (K mod G)-step graph.  EVERY graph the timed
    # region replays is replayed during warm-up first, so no first-replay upload sits inside the region.
    G = min(K, GRAPH_STEPS)
    n_full, rem = divmod(K, G)
    plan = [tuple(i % R for i in range(G))] * n_full + ([tuple((n_full * G + i) % R for i in range(rem))] if rem else [])
    graph_mode = not args.no_graph and not args.no_epoch

    # K <= GRAPH_STEPS: the timed region is ONE graph, and its two events are event-record NODES of that graph
    # (after a 0.1 ms device-side spin), so the K steps are timed on the device without the host -> device
    # latency of the graph launch; stream-recorded events around the replay are kept next to it.
    in_graph_events = graph_mode and len(plan) == 1

    def run_plan():
        if graph_mode:
            for key in plan:
                trainer.run_epoch(key, timed=in_graph_events)
        else:
            for i in range(K):
                trainer.step(i % R)

    warm_steps = 0
    if graph_mode:
        for key in set(plan):
            trainer.capture_epoch(key, timed=in_graph_events)
        while warm_steps < W:
            for key in dict.fromkeys(plan):      # each distinct graph at least once
                trainer.run_epoch(key, timed=in_graph_events)
                warm_steps += len(key)
    else:
        while warm_steps < max(W, R if not args.no_graph else W):
            trainer.step(warm_steps % R)
            warm_steps += 1
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = lib.gad_launch_count()
    clocks.mark(True)
    with torch.cuda.stream(trainer.stream):
        # a short device-side spin BEFORE the first event lets the host enqueue the graph launches while the
        # device is still busy, so the region between the events is device time of the K steps, not launch latency
        torch.cuda._sleep(int(4e5))
    ev0.record(trainer.stream)
    run_plan()
    ev1.record(trainer.stream)
    barrier()
    clocks.mark(False)
    trainer.check_peer()
    # what the last timed step handed back, written before anything below runs more steps on the same buffers
    if args.dump_outputs and rank == 0:
        last = trainer.slots[plan[-1][-1] if graph_mode else (K - 1) % R]
        outputs = {"loss": last.loss, "x_phys": last.x_phys, "params": trainer.flat, "grads": trainer.gflat}
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.detach().cpu().numpy())
    ms_stream_events = ev0.elapsed_time(ev1)
    ms_total = trainer.epoch_elapsed_ms(plan[0]) if in_graph_events else ms_stream_events
    eager_launches = lib.gad_launch_count() - launches0
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / K
    value = world * n_nodes / (ms_step * 1e-3)

    # ---- data-parallel self-check (N > 1): replicas bit-identical, in-kernel exchange == NCCL route ----
    dp_check = None
    if world > 1:
        dp_check = trainer.dp_selfcheck(list(range(min(R, 4))), steps=min(K, 24))

    # kernels per step: counted once from an eager issue of the same step
    l0 = lib.gad_launch_count()
    trainer._issue(s0, trainer.stream.cuda_stream)
    trainer.synchronize()
    launches_per_step = lib.gad_launch_count() - l0
    gpu_launches = int(launches_per_step * K) if not args.no_graph else int(eager_launches)

    # ---- dominant-kernel timing (CUDA events on the launching stream, eager issue) ----------
    from g_adaptivity_b200 import functional as GF
    P = _lib.ptr
    peak, peak_src = measured_peaks()
    ell = GF.use_ell(s0.graph, trainer.CE)
    nk = min(max(K, 20), 200)
    evs = []
    if ell:
        # the step IS one kernel (k_ell_train); time that launch (all-reduce / Adam excluded when N > 1)
        with torch.cuda.stream(trainer.stream):
            torch.cuda._sleep(int(2e7))          # let the host run ahead: event pairs time the device only
            for i in range(nk):
                s = trainer.slots[i % R]
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record(trainer.stream)
                trainer._issue(s, trainer.stream.cuda_stream, stage="pre")
                a1.record(trainer.stream)
                evs.append((a0, a1))
        trainer.synchronize()
        k_iso_ms = statistics.median(a0.elapsed_time(a1) for a0, a1 in evs[5:])
        step_bytes = ab["step_per_node"] * n_nodes
        # One launch per step: the kernel's average launch duration over the timed region is the region's
        # device time (CUDA events on the launching stream) / the launches in it.  Consecutive launches
        # are chained by programmatic dependent launch, so each one's input staging runs in the shadow of
        # its predecessor; the duration of a launch issued alone (no overlap) is reported next to it.
        one_launch = int(launches_per_step) == 1 and not args.no_graph
        k_ms = ms_step if one_launch else k_iso_ms
        achieved = step_bytes / (k_ms * 1e-3) / 1e9
        traffic = ncu_traffic("k_ell_train")
        roofline = {"bound": "hbm", "kernel": "k_ell_train (pack + fwd + loss + bwd + reduce / chain rule / "
                                              + ("peer all-reduce / " if trainer.fused_dp else "") + "Adam / refold tail, one launch)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": step_bytes, "kernel_ms": k_ms,
                    "kernel_ms_isolated": k_iso_ms, "frac_isolated": step_bytes / (k_iso_ms * 1e-3) / 1e9 / peak,
                    "bytes_per_node": ab["step_per_node"],
                    "note": "algorithmic bytes = SURVEY 8(d) streaming model (663 B/node/train call); the mesh-resident "
                            "kernel keeps states in shared memory / L2, so real DRAM traffic (`traffic`) is far lower: "
                            "the kernel is bound by shared-memory gather latency and issue slots, not HBM",
                    "timing": ("kernel_ms = timed region (CUDA events on the launching stream) / launches in it, PDL-chained "
                               "graph replay; " if one_launch else "") +
                              "kernel_ms_isolated = CUDA events around single eager launches after the timed region"}
    else:
        for i in range(nk):
            s = trainer.slots[i % R]
            g = s.graph
            st = trainer.stream.cuda_stream
            with torch.cuda.stream(trainer.stream):
                lib.gad_prepare_weights(P(trainer.Wq), P(trainer.bq), P(trainer.Wk), trainer.Lw, trainer.C, trainer.CE,
                                        model.inv_temp, P(trainer.Mu), st)
                lib.gad_pack_features(P(s.x_comp), P(s.f), P(s.uu), None, None, s.N, model.dim, trainer.CE, P(s.states), st)
                lib.gad_deform_fwd(P(g.rowptr), P(g.col_walk), s.N, g.E, P(g.tile_ptr), g.T, g.max_tile_nodes,
                                   g.max_tile_edges, P(s.states), model.dim, trainer.CE, P(trainer.Mu), trainer.Lw,
                                   P(trainer.tau), trainer.L, 0, P(s.x_phys), P(s.states), P(s.fwd_ws), s.fwd_ws_bytes, st)
                lib.gad_mesh_loss(P(s.x_phys), P(s.target), s.N * model.dim, 0, 1.0 / (s.N * model.dim), P(s.loss),
                                  P(s.g_out), P(s.loss_ws), st)
                b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                b0.record(trainer.stream)
                lib.gad_deform_bwd(P(g.rowptr), P(g.col_walk), P(g.t_rowptr), P(g.t_dst_walk), s.N, g.E, P(g.tile_ptr), g.T,
                                   g.max_tile_nodes, g.max_tile_edges, P(s.states), P(s.g_out), model.dim, trainer.CE,
                                   P(trainer.Mu), trainer.Lw, P(trainer.tau), trainer.L, P(trainer.gMu), P(trainer.gtau),
                                   None, P(s.bwd_ws), s.bwd_ws_bytes, st)
                b1.record(trainer.stream)
            evs.append((b0, b1))
        trainer.synchronize()
        bwd_ms = statistics.median(b0.elapsed_time(b1) for b0, b1 in evs[5:])
        bwd_bytes = ab["bwd_per_node"] * n_nodes
        achieved = bwd_bytes / (bwd_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "k_fused_bwd (+k_fused_reduce)", "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": bwd_bytes, "kernel_ms": bwd_ms,
                    "step_frac": (value / world) * ab["step_per_node"] / 1e9 / peak,
                    "timing": "CUDA events on the launching stream around the kernel, median of eager launches"}

    # ---- end-to-end: pinned host buffers in, loss out, every step --------------------------
    e2e = None
    if not args.skip_e2e:
        ke = min(max(K, 400), 2000)      # the pipeline needs a few steps to fill: never fewer than 400
        # host side of the public API: every batch packed once into ONE pinned buffer in the slot's input
        # layout (DeformerTrainer.pack_host), so a step's inputs travel host -> device in a single copy.
        # The synthetic dataset is on one shared mesh (as the reference's `randg` datasets, src/data.py:143):
        # x_comp is resident per slot and the per-step copy is the per-sample part, target | f | uu.
        packed = [trainer.pack_host(r, host_batches[r], with_x_comp=False, write_combined=args.write_combined)
                  for r in range(R)]
        relay, path_rates, relay_trials = None, None, None
        # the relay lives in the native loop (graph replay of the one-launch step; the route is agreed across ranks)
        native_loop = trainer.use_graph and all(trainer._one_launch(s) for s in trainer.slots)
        if world > 1 and args.relay == "auto" and native_loop:
            # Unequal host->device paths (DESIGN section 15): a probe proposes pairs and a fraction; the proposal, its
            # mirror image and the direct loop are then TIMED on the real loop (short trials, max over ranks) and the
            # fastest is kept -- the probe alone has been wrong about the direction.
            from g_adaptivity_b200 import dp as gdp
            try:
                _, path_rates = gdp.balance_host_paths(dev)
                plans = {"direct": {}}
                if path_rates is not None:
                    devs = list(range(world))
                    fwd = gdp.plan_host_relays(path_rates, devs)
                    if fwd:
                        plans["probe"] = fwd
                        plans["mirror"] = {via: (q, y) for q, (via, y) in fwd.items()}
                    # a prior from the boxes measured so far (profiles/r02_h2d_probe_8gpu.json: the lower half of the
                    # GPUs has the slower paths, 21 against 37 GB/s, i.e. y = 0.27), and its mirror image; like every
                    # proposal it only survives if the timed trial says so
                    if world >= 2 and world % 2 == 0:
                        h = world // 2
                        plans["halves"] = {q: (q + h, 0.27) for q in range(h)}
                        plans["halves_mirror"] = {q + h: (q, 0.27) for q in range(h)}
                if os.environ.get("GAD_RELAY_PLAN"):       # testing aid: "rank:device:fraction,..." as the only proposal
                    forced = {}
                    for item in os.environ["GAD_RELAY_PLAN"].split(","):
                        q, via, y = item.split(":")
                        forced[int(q)] = (int(via), float(y))
                    plans = {"direct": {}, "forced": forced}
                relay_trials = {}
                trainer.run_from_host(packed, 2 * R)
                nbytes = packed[0].numel() * 4
                for name, plan in plans.items():
                    cand = plan.get(rank)
                    # set-up (context + staging on the partner GPU, peer access) may fail on ONE rank only: agree on
                    # it before any rank enters a loop whose steps exchange gradients with the others
                    ok = 1.0
                    try:
                        if cand is not None:
                            trainer._relay_descriptor(cand, nbytes, R)
                    except Exception:      # noqa: BLE001
                        ok = 0.0
                    okt = torch.tensor([ok], dtype=torch.float64, device=dev)
                    dist.all_reduce(okt, op=dist.ReduceOp.MIN)
                    if float(okt.item()) < 1.0:
                        relay_trials[name] = "set-up failed on a rank"
                        continue
                    trainer.run_from_host(packed, 2 * R, relay=cand)          # warm the candidate's path
                    barrier()
                    t1 = time.perf_counter()
                    trainer.run_from_host(packed, 120, relay=cand)
                    barrier()
                    tt1 = torch.tensor([time.perf_counter() - t1], dtype=torch.float64, device=dev)
                    dist.all_reduce(tt1, op=dist.ReduceOp.MAX)
                    relay_trials[name] = float(tt1.item()) / 120
                timed = {k: v for k, v in relay_trials.items() if isinstance(v, float)}
                best = min(timed, key=timed.get)
                if best != "direct" and timed[best] < 0.97 * timed["direct"]:
                    relay = plans[best].get(rank)
                    relay_trials["chosen"] = best
                else:
                    relay_trials["chosen"] = "direct"
            except Exception as e:      # noqa: BLE001 -- the direct loop always works
                relay, relay_trials = None, {"error": repr(e)[:200]}
            # one more agreement: a rank that fell out of the selection makes everybody run the direct loop
            okt = torch.tensor([0.0 if (relay_trials or {}).get("error") else 1.0], dtype=torch.float64, device=dev)
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            if float(okt.item()) < 1.0:
                relay = None
        trainer.run_from_host(packed, min(2 * R, ke), relay=relay)
        barrier()
        t0 = time.perf_counter()
        losses = trainer.run_from_host(packed, ke, relay=relay)
        barrier()
        dt = time.perf_counter() - t0
        assert losses.numel() == ke and bool(torch.isfinite(losses).all())
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": world * n_nodes * ke / dt, "unit": UNIT, "h2d_bytes_per_step": int(s0.h2d_bytes),
               "d2h_bytes_per_step": 4, "ms_per_step": 1e3 * dt / ke, "steps": ke,
               "h2d_gb_per_s_per_rank": s0.h2d_bytes * ke / dt / 1e9,
               "api": "DeformerTrainer.run_from_host over pack_host buffers (loop in the C library, gad_pipeline_run): "
                      "per step ONE pinned H2D copy of the per-sample inputs target|f|uu (16 B/node; x_comp of the "
                      "shared mesh is resident) on a copy stream, overlapped with the previous step's kernel; graph "
                      "replay of the one-launch step; async D2H of the loss",
               "cpu_affinity": affinity, "host_memory": "pinned, write-combined" if args.write_combined else "pinned"}
        if world > 1:
            mine = torch.tensor([-1.0, 0.0] if relay is None else [float(relay[0]), float(relay[1])],
                                dtype=torch.float64, device=dev)
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            e2e["host_paths"] = {
                "gb_s_per_rank_under_load": None if path_rates is None else [round(x, 1) for x in path_rates],
                "relay": {str(q): {"via_device": int(a[0]), "fraction": round(float(a[1]), 3)}
                          for q, a in enumerate(allr) if a[0] >= 0},
                "trials_ms_per_step": None if relay_trials is None else
                {k: (round(1e3 * v, 4) if isinstance(v, float) else v) for k, v in relay_trials.items()},
                "what": "ranks whose host->device path is slower under load send that fraction of every batch through "
                        "the partner GPU (host -> staging there, then NVLink): gad_pipeline_run_relay"}

    clk = clocks.stop() if rank == 0 else None

    # ---- the other BASELINE configs, device-timed (cfg 2 stays `value`) ---------------------------
    configs = None
    if not args.skip_configs:
        configs = {}
        it = 5 if K <= 50 else 20
        try:
            configs["cfg5_50x50_global_batch_8192_train"] = time_cfg5(dev, rank, world, max(3, it // 2), peak, barrier)
        except Exception as e:      # noqa: BLE001 -- the headline line must survive a failing extra
            if world > 1:
                raise
            configs["cfg5_50x50_global_batch_8192_train"] = {"error": repr(e)[:300]}
        if world == 1:
            for name, fn in (
                    ("cfg1_15x15_single_mesh_fwd", lambda: time_forward_config(dev, (15, 15), 1, {}, False, it, peak)),
                    ("cfg3_burgers_1d_200_batch_4096_fwd",
                     lambda: time_forward_config(dev, (200,), 4096, {}, True, it, peak)),
                    ("cfg4_200x200_64_rk4_steps_fwd",
                     lambda: time_forward_config(dev, (200, 200), 1, {"ode_method": "rk4", "num_layers": 64}, False, it, peak)),
                    ("f1_pde_loss_2d_cfg2_shape_train_step", lambda: time_pde_loss_2d(dev, 3)),
                    ("cfg2_reference_loop_shape", lambda: time_loop_shape(dev, 20))):
                try:
                    configs[name] = fn()
                except Exception as e:      # noqa: BLE001
                    configs[name] = {"error": repr(e)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:      # reported at N = 1 only (the other ranks would spin)
        r = time_cpu_oracle(steps=20, warmup=1, budget_s=20.0)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
               "ms_per_step": r["ms_per_step"]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": WORKLOAD,
                "gradient_exchange": (None if world == 1 else ("all-reduce inside the train kernel over NVLink peer memory"
                                                               if trainer.fused_dp else "NCCL all-reduce")),
                "nodes_per_step_per_gpu": n_nodes, "edges_per_step_per_gpu": n_edges, "live_channels": model.live,
                "l2": f"ring of {R} distinct resident batches, {ro_bytes / 1e6:.0f} MB of read-only per-step inputs walked "
                      "in order (> 126 MB L2: no step finds its inputs cached)",
                "topology": ("shared: one ELL table per tile shape (dataset on one mesh), graph built for one tile"
                             if s0.graph.uniform else "general: ELL rows for every node of the batch"),
                "launch": "eager" if args.no_graph else ("cuda-graph replay, one graph per step" if args.no_epoch else
                                                         f"cuda-graph replay: {n_full} x one graph of {G} steps"
                                                         + (f" + one graph of {rem} steps" if rem else "")
                                                         + ", programmatic dependent launch between steps; every graph "
                                                           "replayed during warm-up"),
                "warmup_steps_run": warm_steps,
                "timing": ("CUDA events recorded as nodes of the K-step graph (device time of the K steps); the same "
                           f"region between stream-recorded events around the replay: {ms_stream_events / K * 1e3:.2f} us/step "
                           "(adds the device-side start-up of the graph launch and a 0.1 ms spin)"
                           if in_graph_events else "CUDA events recorded on the launching stream around the replays"),
                "tiles": s0.graph.T, "max_tile_nodes": s0.graph.max_tile_nodes,
            },
            "clocks": clk, "e2e": e2e, "gpu_launches": gpu_launches, "launches_per_step": int(launches_per_step),
            "roofline": roofline, "cpu_baseline": cpu,
        }
        if dp_check is not None:
            line["dp_check"] = dp_check
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave without tearing NCCL down: the captured graphs hold collectives and
        # destroy_process_group() can wait on them forever.  Everything is flushed; the ranks agree
        # that they are done, then exit hard.
        trainer.close()
        dist.barrier()
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        sys.stderr.flush()
        ok = dp_check is None or (dp_check["ranks_equal"] and dp_check["vs_nccl"] == "bit-exact"
                                  and dp_check["parameters_moved"])
        os._exit(0 if ok else 1)


if __name__ == "__main__":
    main()
