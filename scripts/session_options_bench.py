#!/usr/bin/env python
"""Forward of models with global CNN features, gnn_normalize or the learnable temperature: the module call against
the CUDA-graph replay of `model.inference_session(data)`, device-timed, with a bit-for-bit check of the replay.

    python scripts/session_options_bench.py [--iters 50] [--rounds 3] [--out FILE.json]

Workloads (inputs device-resident, `model(data)` under no_grad with gad_sync_timestamp=False so that no call waits
for the stream):
  glob_256x30x30       256 meshes of 30x30, gnn_inc_glob_feat_f and _uu (default model otherwise);
  glob_uu_4096x200     the Burgers preset on 4096 1-D meshes of 200 nodes with gnn_inc_glob_feat_uu;
  glob_cluster_1x64x64 one 64x64 mesh with both CNNs, forward on the cluster kernel (GAD_FWD_POLICY=cluster);
  normalize_4096x200   the Burgers preset (BASELINE cfg 3 shape) with gnn_normalize;
  learnable_a_256x30x30  256 meshes of 30x30 with softmax_temp_type='learnable_a'.
Per workload, `rounds` alternations of: the module call with the default alpha policy (the model keeps the layer
states conv.stored_alpha reads), the module call with gad_store_alpha=False (the graph policy global-feature models
had before they kept alpha; the difference is what keeping it costs), and the session replay with a new `uu` copied
in each call (`sess(uu=...)`, host-paced, CUDA events around `iters` calls).  `device_replay_us`: the graph replayed
back to back behind a device spin, CUDA events around each replay (no host time in it).  The best round of each is
reported.  `bit_equal`: a replay with a fresh uu equals `model(data)` on a batch carrying it (torch.equal).
The card name, power limit and maximum SM clock are printed with the numbers (nvidia-smi).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from g_adaptivity_b200 import GNN, synth  # noqa: E402

FU = {"gnn_inc_glob_feat_f": True, "gnn_inc_glob_feat_uu": True}
WORKLOADS = {
    # name: mesh dims, meshes, Burgers preset, options, environment
    "glob_256x30x30": ((30, 30), 256, False, FU, {}),
    "glob_uu_4096x200": ((200,), 4096, True, {"gnn_inc_glob_feat_uu": True}, {}),
    "glob_cluster_1x64x64": ((64, 64), 1, False, FU, {"GAD_FWD_POLICY": "cluster"}),
    "normalize_4096x200": ((200,), 4096, True, {"gnn_normalize": True}, {}),
    "learnable_a_256x30x30": ((30, 30), 256, False, {"softmax_temp_type": "learnable_a"}, {}),
}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    return q.stdout.strip()


def make(md, B, burgers, over, dev):
    opt = synth.burgers_opt(md) if burgers else synth.default_opt(md)
    opt.update(device=str(dev), gad_sync_timestamp=False, **over)
    ds = synth.SyntheticDataset(len(md), md)
    ds.x_comp_shared = synth.make_batch(md, 1).x_comp
    torch.manual_seed(42)
    model = GNN(ds, opt).to(dev).eval()
    data = synth.make_batch(md, B, seed=0, burgers=burgers).to(dev)
    return model, data


def module_us(model, data, store_alpha, iters):
    model.opt["gad_store_alpha"] = store_alpha
    for _ in range(3):
        model(data)
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        model(data)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    model.opt["gad_store_alpha"] = True
    return 1000.0 * statistics.median(ts)


def session_us(sess, uu, iters):
    for _ in range(3):
        sess(uu=uu)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        sess(uu=uu)
    e1.record()
    torch.cuda.synchronize()
    return 1000.0 * e0.elapsed_time(e1) / iters


def device_replay_us(sess, iters):
    pairs = []
    with torch.cuda.stream(sess.stream):
        torch.cuda._sleep(int(4e7))
        for _ in range(iters):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(sess.stream)
            sess.cuda_graph.replay()
            a1.record(sess.stream)
            pairs.append((a0, a1))
    sess.stream.synchronize()
    return 1000.0 * statistics.median(a0.elapsed_time(a1) for a0, a1 in pairs[2:])


def route(model):
    g = model.last_graph
    if g.tile_ptr is not None:
        return "mesh-resident"
    return "cluster" if getattr(g, "clf_in", None) is not None and not g.stream_fwd_preferred(
        model.CE, model.opt["num_layers"] * (4 if model.opt.get("ode_method") == "rk4" else 1)) else "stream"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("session_options_bench.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    info = card()
    print(f"# {info}", flush=True)
    rows = []
    names = args.only.split(",") if args.only else list(WORKLOADS)
    for name in names:
        md, B, burgers, over, envd = WORKLOADS[name]
        saved = {k: os.environ.get(k) for k in envd}
        os.environ.update(envd)
        try:
            model, data = make(md, B, burgers, over, dev)
            with torch.no_grad():
                model(data)
                sess = model.inference_session(data)
                g = torch.Generator(device="cpu").manual_seed(1)
                uu = (data.uu_tensor * (1.0 + 0.3 * torch.rand(data.uu_tensor.shape, generator=g).to(dev))).contiguous()
                got = sess(uu=uu).clone()
                data.uu_tensor = uu
                bit_equal = bool(torch.equal(got, model(data)))
                t = {"alpha": [], "no_alpha": [], "session": [], "device": []}
                for _ in range(args.rounds):
                    t["alpha"].append(module_us(model, data, True, args.iters))
                    t["no_alpha"].append(module_us(model, data, False, args.iters))
                    t["session"].append(session_us(sess, uu, args.iters))
                    t["device"].append(device_replay_us(sess, args.iters))
            row = dict(workload=name, nodes=int(data.x_comp.shape[0]), route=route(model),
                       n_glob_used=model.n_glob_used, bit_equal=bit_equal,
                       module_us=round(min(t["alpha"]), 1), module_no_alpha_us=round(min(t["no_alpha"]), 1),
                       session_us=round(min(t["session"]), 1), device_replay_us=round(min(t["device"]), 1),
                       rounds={k: [round(x, 1) for x in v] for k, v in t.items()})
            rows.append(row)
            print(json.dumps(row), flush=True)
            del sess, model, data
            torch.cuda.empty_cache()
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump({"card": info, "iters": args.iters, "rounds": args.rounds, "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
