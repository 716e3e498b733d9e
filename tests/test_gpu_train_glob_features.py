"""DeformerTrainer on models with global CNN features (gnn_inc_glob_feat_f / _uu, src/GNN.py:242-268).

A step on such a batch is the CNN forward (csrc/glob_cnn.cu), the per-mesh bias offset du (csrc/glob_train.cu), the
mesh-resident deformer forward and backward with du, the adjoint of du (CNN cotangents and the du terms of gWq / gWk),
the CNN backward into the flat gradient and Adam over the whole flat vector.  Bars are tests/test_glob_features.py's:
coordinates 1e-5 and gradients 2e-4 against the fp64 oracle; after Adam steps the project's Adam bar (2e-3 of the
largest parameter, lin_key.bias excluded: its gradient is analytically zero, so Adam turns rounding noise into O(lr)).
"""
import copy
import json
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

import gad_testutil as util
from g_adaptivity_b200 import _lib, synth
from g_adaptivity_b200.trainer import DeformerTrainer
from oracle import gnn_oracle
from test_glob_features import NAMES, _check_against, _dataset, _load
from test_gpu_parity import cuda_model

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ROWS_2D = [
    ((12, 12), 5, {"gnn_inc_glob_feat_f": True, "gnn_inc_glob_feat_uu": True}),
    ((30, 30), 3, {"gnn_inc_glob_feat_f": True, "gnn_inc_glob_feat_uu": True, "hidden_dim": 16}),
    ((9, 9), 4, {"gnn_inc_glob_feat_uu": True, "share_conv": False, "num_layers": 3}),
    ((10, 10), 3, {"gnn_inc_glob_feat_f": True, "ode_method": "rk4", "num_layers": 2}),
    ((8, 8), 2, {"gnn_inc_glob_feat_f": True, "hidden_dim": 4}),          # nothing global survives the truncation
]


def _case_2d(md, B, over, seed=9):
    opt = synth.default_opt(md, **over)
    ds = _dataset(md)
    data = synth.make_batch(md, B, seed=seed)
    torch.manual_seed(42)
    state = copy.deepcopy(gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict())
    return opt, ds, data, state


def _case_fixture(name):
    fx = _load(name)
    md = fx["mesh_dims_list"][0]
    return util.fixture_opt(fx), _dataset(md), util.fixture_batch(fx), fx["state_dict"]


def _step_without_optimizer(tr, sid):
    with torch.cuda.stream(tr.stream):
        tr._issue(tr.slots[sid], tr.stream.cuda_stream, with_optimizer=False)
    tr.synchronize()
    return tr.slots[sid].loss.item()


def _oracle64(ds, opt, data, state):
    ref = gnn_oracle.GNNRef(ds, copy.deepcopy(opt))
    ref.load_state_dict(state)
    ref = ref.double()
    d64 = data.clone()
    for k in d64.keys():
        v = getattr(d64, k)
        if torch.is_tensor(v) and v.dtype == torch.float32:
            setattr(d64, k, v.double())
    out = ref(d64)
    loss = gnn_oracle.mesh_loss(out, d64.x_phys)
    loss.backward()
    return out, loss.item(), {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}


# 1 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [("2d", i) for i in range(len(ROWS_2D))] + [("fixture", n) for n in NAMES],
                         ids=[f"2d-{r[0][0]}x{r[0][1]}-B{r[1]}-{i}" for i, r in enumerate(ROWS_2D)] + NAMES)
def test_one_step_matches_the_fp64_oracle(case):
    kind, key = case
    opt, ds, data, state = _case_2d(*ROWS_2D[key]) if kind == "2d" else _case_fixture(key)
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert s.glob == (model.n_glob_used > 0) and tr._one_launch(s) == (not s.glob)
    loss = _step_without_optimizer(tr, sid)
    out64, l64, g64 = _oracle64(ds, opt, data, state)
    assert util.rel_err(s.x_phys, out64.reshape(s.x_phys.shape)) <= 1e-5
    assert abs(loss - l64) <= 1e-5 * abs(l64), (loss, l64)
    if model.n_glob_used == 0:
        # a plain deformer: the CNNs stay out of the flat vector and get no gradient, as on the module path
        assert all(p.grad is None for n, p in model.named_parameters() if "global_feature" in n)
        g64 = {n: g for n, g in g64.items() if "global_feature" not in n}
    else:
        assert s.graph.T == len(s.graph.mesh_sizes)                             # one mesh per tile
    _check_against(model, g64)


# 2 ------------------------------------------------------------------------------------------------------------------
K, LR = 10, 1e-2


def _module_adam(ds, opt, state, batches, loss_fn):
    lossf = F.l1_loss if loss_fn == "l1" else F.mse_loss
    m = cuda_model(ds, opt, state)
    m.train()
    optim = torch.optim.Adam(m.parameters(), lr=LR)
    losses = []
    for k in range(K):
        data = batches[k % len(batches)]
        optim.zero_grad(set_to_none=True)
        out = m(data)
        loss = lossf(out, data.x_phys.cuda().reshape(out.shape))
        loss.backward()
        optim.step()
        losses.append(float(loss.item()))
    return {n: p.detach().cpu().clone() for n, p in m.named_parameters()}, losses


def _trainer_adam(ds, opt, state, batches, loss_fn, mode):
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, lr=LR, loss_fn=loss_fn, use_cuda_graph=(mode != "eager"))
    sids = [tr.add_batch(b) for b in batches]
    losses = []
    if mode == "epoch":
        for _ in range(K // len(sids)):
            tr.run_epoch(sids)
            tr.synchronize()
            losses += [float(tr.slots[s].loss.item()) for s in sids]
    else:
        for k in range(K):
            l = tr.step(sids[k % len(sids)])
            tr.synchronize()
            losses.append(float(l.item()))
    assert int(tr.step_count.item()) == K
    return tr, {n: p.detach().cpu().clone() for n, p in model.named_parameters()}, losses


def _compare_params(got, want, losses, ref_losses, tol=2e-3):
    assert sorted(got) == sorted(want)
    names = [n for n in want if "lin_key.bias" not in n]
    scale = max(want[n].abs().max().item() for n in names)
    worst = max((got[n] - want[n]).abs().max().item() for n in names) / scale
    print(f"parameters after {K} Adam steps: max |trainer - module| / max |param| = {worst:.3e}")
    assert worst <= tol, worst
    assert abs(losses[0] - ref_losses[0]) <= 1e-5 * abs(ref_losses[0])
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 2e-3 * abs(b), (losses, ref_losses)


@pytest.fixture(scope="module")
def small_case():
    md = (12, 12)
    opt = synth.default_opt(md, lr=LR, gnn_inc_glob_feat_f=True, gnn_inc_glob_feat_uu=True)
    ds = _dataset(md)
    batches = [synth.make_batch(md, 8, seed=31, first_mesh_id=r * 8) for r in range(2)]
    torch.manual_seed(42)
    state = copy.deepcopy(gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict())
    want, ref_losses = _module_adam(ds, opt, state, batches, "l1")
    return opt, ds, batches, state, want, ref_losses


@pytest.mark.parametrize("mode", ["eager", "graph", "epoch"])
def test_k_adam_steps_match_the_module_path(small_case, mode):
    opt, ds, batches, state, want, ref_losses = small_case
    tr, got, losses = _trainer_adam(ds, opt, state, batches, "l1", mode)
    assert any("global_feature" in n for n in got)
    _compare_params(got, want, losses, ref_losses)


@pytest.mark.parametrize("md,B,loss_fn", [((30, 30), 256, "l1"), ((200,), 4096, "l1"), ((200,), 4096, "mse")])
def test_k_adam_steps_match_the_module_path_at_production_shapes(md, B, loss_fn):
    if len(md) == 2:
        opt = synth.default_opt(md, lr=LR, gnn_inc_glob_feat_f=True)
    else:
        opt = synth.burgers_opt(md, lr=LR, gnn_inc_glob_feat_f=True, gnn_inc_glob_feat_uu=True)
    ds = _dataset(md)
    batches = [synth.make_batch(md, B, seed=5, burgers=len(md) == 1)]
    torch.manual_seed(42)
    state = copy.deepcopy(gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict())
    want, ref_losses = _module_adam(ds, opt, state, batches, loss_fn)
    tr, got, losses = _trainer_adam(ds, opt, state, batches, loss_fn, "graph")
    assert tr.slots[0].glob
    _compare_params(got, want, losses, ref_losses)


# 3 ------------------------------------------------------------------------------------------------------------------
def test_steps_are_bit_reproducible(small_case):
    opt, ds, batches, state, _, _ = small_case
    runs = [_trainer_adam(ds, opt, state, batches, "l1", "graph") for _ in range(2)]
    assert runs[0][2] == runs[1][2] and torch.equal(runs[0][0].flat, runs[1][0].flat)


# 4 ------------------------------------------------------------------------------------------------------------------
def test_train_batch_and_run_from_host_equal_resident_steps(small_case):
    opt, ds, _, state, _, _ = small_case
    md = (12, 12)
    fresh = [synth.make_batch(md, 6, seed=50 + k) for k in range(4)]
    for b in fresh:
        b.pin_memory()
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, lr=LR)
    got = []
    for b in fresh:
        got.append(float(tr.train_batch(b).item()))
        tr.synchronize()
    model2 = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr2 = DeformerTrainer(model2, lr=LR)
    sids = [tr2.add_batch(b) for b in fresh]
    want = []
    for sid in sids:
        want.append(float(tr2.step(sid).item()))
        tr2.synchronize()
    assert got == want and torch.equal(tr.flat, tr2.flat)

    batches = fresh[:2]
    outs = []
    for mode in ("resident", "packed_native", "python_loop"):
        model = cuda_model(ds, opt, state, gad_store_alpha=False)
        tr = DeformerTrainer(model, lr=LR)
        sids = [tr.add_batch(b) for b in batches]
        if mode == "resident":
            losses = []
            for k in range(6):
                l = tr.step(sids[k % 2])
                with torch.cuda.stream(tr.stream):
                    losses.append(l.clone())
            tr.synchronize()
            losses = torch.stack([x.cpu() for x in losses]).reshape(-1)
        elif mode == "packed_native":
            src = [tr.pack_host(sid, b) for sid, b in zip(sids, batches)]
            losses = tr.run_from_host(src, 6, native=True).clone()
        else:
            losses = tr.run_from_host(batches, 6, native=False).clone()
        outs.append((losses, tr.flat.clone().cpu()))
    for losses, flat in outs[1:]:
        assert torch.equal(outs[0][0], losses) and torch.equal(outs[0][1], flat)


# 5 ------------------------------------------------------------------------------------------------------------------
def test_refusals():
    opt = synth.default_opt((6, 6), gnn_inc_glob_feat_f=True)
    model = cuda_model(_dataset((6, 6)), opt)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    with pytest.raises(NotImplementedError, match="equal size"):
        tr.add_batch(synth.make_mixed_batch([(6, 6), (7, 7)], seed=1))
    opt = synth.default_opt((60, 60), gnn_inc_glob_feat_f=True)
    model = cuda_model(_dataset((60, 60)), opt)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    with pytest.raises(NotImplementedError, match="mesh-resident"):
        tr.add_batch(synth.make_batch((60, 60), 2, seed=1))
    opt = synth.default_opt((7, 7), gnn_inc_glob_feat_f=True, softmax_temp_type="learnable_a")
    with pytest.raises(NotImplementedError):
        DeformerTrainer(cuda_model(_dataset((7, 7)), opt))


# 6 ------------------------------------------------------------------------------------------------------------------
def test_c_abi_rejects_bad_arguments():
    lib = _lib.load()
    buf, out = torch.zeros(4096, device="cuda"), torch.zeros(64, device="cuda")
    p = buf.data_ptr()
    # (B, Co, n_g, Lw, C, z0, live, CE)
    good = (2, 4, 3, 1, 8, 3, 4, 4)
    bad = [((2, 4, 0, 1, 8, 3, 4, 4), "n_g"), ((2, 4, 9, 1, 8, 3, 4, 4), "n_g"),
           ((2, 4, 3, 1, 8, 6, 4, 4), "z0"), ((2, 4, 3, 1, 8, 3, 5, 4), "live")]

    def fwd(B, Co, n_g, Lw, C_, z0, live, CE, g_uu=p):
        return lib.gad_glob_bias_fwd(p, g_uu, B, Co, n_g, p, p, Lw, C_, z0, live, CE, 1.0, out.data_ptr(), None)

    for args, word in bad:
        assert fwd(*args) != 0
        assert word in lib.gad_last_error().decode()
    assert fwd(2, 4, 5, 1, 8, 3, 4, 4, g_uu=None) != 0          # 5 channels from one output of 4
    assert fwd(*good) == 0
    B, Co, n_g, Lw, C_, z0, live, CE = good
    rc = lib.gad_glob_bias_bwd(p, p, B, Co, n_g, p, p, Lw, C_, z0, live, CE, 1.0, p, 16, p, p, p, p, None)
    assert rc != 0 and "workspace" in lib.gad_last_error().decode()
    assert lib.gad_absmax(p, 0, p, None) != 0
    torch.cuda.synchronize()


# 7 ------------------------------------------------------------------------------------------------------------------
def test_loopback_slot_takes_the_nccl_route():
    opt = synth.default_opt((12, 12), gnn_inc_glob_feat_f=True)
    model = cuda_model(_dataset((12, 12)), opt, gad_store_alpha=False, gad_peer_loopback=(2, 1))
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(synth.make_batch((12, 12), 4, seed=3))
    assert tr.slots[sid].glob and not tr.slots[sid].peer_route and not tr._one_launch(tr.slots[sid])


@pytest.mark.timeout(300)
def test_two_gpus_match_one_gpu_on_the_union_batch(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, B, steps = 2, 4, 6
    out = tmp_path / "dp_glob.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29537", os.path.join(ROOT, "tests", "dp_glob_worker.py"),
           str(out), str(steps), str(B)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads(out.read_text())
    assert res["ranks_equal"] and not res["peer_route"] and res["selfcheck"]["ranks_equal"]
    md = (12, 12)
    opt = synth.default_opt(md, lr=LR, gnn_inc_glob_feat_f=True, gnn_inc_glob_feat_uu=True)
    torch.manual_seed(42)
    model = cuda_model(_dataset(md), opt, gad_store_alpha=False)
    tr = DeformerTrainer(model, lr=LR)
    sids = [tr.add_batch(synth.make_batch(md, world * B, seed=7, first_mesh_id=k * world * B)) for k in range(2)]
    for k in range(steps):
        tr.step(sids[k % 2])
    tr.synchronize()
    want = tr.flat.cpu()
    got = torch.tensor(res["flat"])
    live = torch.ones(want.numel(), dtype=torch.bool)
    o = (tr.bk.data_ptr() - tr.flat.data_ptr()) // 4
    live[o:o + tr.bk.numel()] = False            # lin_key.bias: analytically zero gradient
    err = (got - want)[live].abs().max().item() / want[live].abs().max().item()
    assert err <= 2e-3, err
