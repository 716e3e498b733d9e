"""DeformerTrainer with loss_type='modular': the cotangent of x_phys comes from the caller (src/run_GNN.py:111-131).

The reference's loop takes `(loss, x_grads)` from an outside function of the detached x_phys and back-propagates the
pseudo-loss sum(x_phys * x_grads).  The trainer runs that as `forward(sid)` -> the caller's x_grads ->
`step(sid, cotangent=x_grads)`: the loss stages of the training kernels take loss kind 2 (the slot's target rows hold
the cotangent, dL/dx_phys = grad_scale * c with grad_scale = 1, loss = <x_phys, c>), on every route.

Checked: fed the cotangent the L1 / MSE loss stage forms, five Adam steps equal a loss_fn='l1' / 'mse' trainer's bit for
bit on every route; forward(sid)'s x_phys is the step's bit for bit; with a nonlinear outside loss, one step's gradient
matches autograd through the fp64 oracle at the bars of test_gpu_train_rk4 and K Adam steps match model + autograd +
torch.optim.Adam at the Adam bar of test_gpu_train_glob_features; graph replay, determinism, the data-parallel routes
and the refusals."""
import copy
import ctypes
import json
import os
import subprocess
import sys

import pytest
import torch

import gad_testutil as util
from g_adaptivity_b200 import _lib, dp, synth
from g_adaptivity_b200.trainer import DeformerTrainer
from oracle import gnn_oracle
from test_glob_features import _dataset
from test_gpu_parity import cuda_model, grads_of, oracle_model

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LR, STEPS = 1e-2, 5

# route -> (mesh dims, meshes, options, trainer-only options, the route's check)
ROUTES = {
    "euler_one_launch": ((30, 30), 8, {}, {}, lambda tr, s: tr._fused_ell(s)),
    "rk4_one_launch": ((30, 30), 8, {"ode_method": "rk4"}, {}, lambda tr, s: tr._fused_ell(s) and s.rk4_fused),
    "cluster": ((64, 64), 4, {}, {}, lambda tr, s: tr._cluster(s)),
    "stream": ((30, 30), 8, {}, {"gad_force_stream": True}, lambda tr, s: not tr._one_launch_local(s) and not s.chain),
    "rk4_chain": ((50, 50), 4, {"ode_method": "rk4"}, {}, lambda tr, s: not tr._one_launch_local(s) and not s.chain),
    "glob_features": ((12, 12), 5, {"gnn_inc_glob_feat_f": True, "gnn_inc_glob_feat_uu": True}, {},
                      lambda tr, s: s.glob and s.chain),
    "learnable_temp": ((12, 12), 5, {"softmax_temp_type": "learnable_a"}, {}, lambda tr, s: s.temp and s.chain),
    "gnn_normalize": ((12, 12), 5, {"gnn_normalize": True}, {}, lambda tr, s: s.norm and tr._one_launch(s)),
}


def _case(route, seed=5):
    md, B, over, extra, _ = ROUTES[route]
    opt = synth.default_opt(md, **over)
    ds = _dataset(md) if "gnn_inc_glob_feat_f" in over else synth.SyntheticDataset(len(md), md)
    data = synth.make_batch(md, B, seed=seed)
    torch.manual_seed(42)
    state = copy.deepcopy(gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict())
    return opt, ds, data, state, extra


def _trainer(ds, opt, state, loss_fn=None, use_graph=False, **extra):
    """A trainer on `opt`; without loss_fn in the cotangent mode (loss_type='modular')."""
    if loss_fn is None:
        opt = dict(opt, loss_type="modular")
    model = cuda_model(ds, opt, state, gad_store_alpha=False, **extra)
    return model, DeformerTrainer(model, lr=LR, loss_fn=loss_fn, use_cuda_graph=use_graph)


def _mesh_cotangent(x, target, loss_fn, scale):
    """The cotangent the L1 / MSE loss stage forms: sign(x - t) * s, (x - t) * (2 s) (2 s is exact)."""
    d = x - target
    return torch.sign(d) * scale if loss_fn == "l1" else d * (2.0 * scale)


def _state(tr):
    return [t.detach().clone() for t in (tr.flat, tr.exp_avg, tr.exp_avg_sq, tr.step_count)]


def _smooth_grad_fn(target):
    """A nonlinear outside loss of x_phys and its gradient (autograd), as the reference's gradient functions return."""
    def grad_fn(x):
        xd = x.detach().clone().requires_grad_(True)
        loss = _smooth_loss(xd, target)
        g, = torch.autograd.grad(loss, xd)
        return loss.detach(), g
    return grad_fn


def _smooth_loss(x, target):
    d = x - target.to(x.dtype).reshape(x.shape)
    return torch.sqrt((d * d).sum(-1) + 1e-3).mean() + 0.5 * torch.tanh(3.0 * x).pow(2).mean()


# 1, 2 ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("loss_fn", ["l1", "mse"])
@pytest.mark.parametrize("route", list(ROUTES))
def test_mesh_loss_cotangent_trains_bit_for_bit(route, loss_fn):
    """The cotangent of the L1 / MSE loss, built with torch from forward(sid)'s x_phys: five Adam steps give the
    parameters, Adam moments and step count of a loss_fn trainer on the same batch bit for bit, and forward(sid)'s
    x_phys equals what both steps write."""
    opt, ds, data, state, extra = _case(route)
    _, ref = _trainer(ds, opt, state, loss_fn=loss_fn, **extra)
    _, tr = _trainer(ds, opt, state, **extra)
    sr, sc = ref.add_batch(data), tr.add_batch(data)
    s = tr.slots[sc]
    assert ROUTES[route][4](tr, s) and ROUTES[route][4](ref, ref.slots[sr])
    target = ref.slots[sr].target
    scale = dp.local_grad_scale(s.N * tr.dim, s.count_global)
    for _ in range(STEPS):
        x = tr.forward(sc).clone()
        ref.step(sr)
        ref.synchronize()
        assert torch.equal(x, ref.slots[sr].x_phys)
        tr.step(sc, cotangent=_mesh_cotangent(x, target, loss_fn, scale))
        tr.synchronize()
        assert torch.equal(s.x_phys, x)
    for a, b in zip(_state(tr), _state(ref)):
        assert torch.equal(a, b)
    assert int(tr.step_count.item()) == STEPS
    # the step's loss is the pseudo-loss <x_phys, c> of its last cotangent
    c = _mesh_cotangent(x, target, loss_fn, scale).double()
    want = (x.double() * c).sum().item()
    assert abs(tr.slots[sc].loss.item() - want) <= 1e-5 * max(abs(want), (x.double().abs() * c.abs()).sum().item())


# 3 ------------------------------------------------------------------------------------------------------------------
def _oracle_grads(ds, opt, data, state):
    """Gradients of sum(x_phys * x_grads(x_phys)) through the oracle in fp64, with the fp32 oracle's deviations from
    them (the conditioning floor of gad_testutil.check_grads_conditioned)."""
    res = []
    for double in (False, True):
        ref = oracle_model(ds, opt, state)
        d = data.clone()
        if double:
            ref = ref.double()
            for k in d.keys():
                v = getattr(d, k)
                if torch.is_tensor(v) and v.dtype == torch.float32:
                    setattr(d, k, v.double())
        out = ref(d)
        _, g = _smooth_grad_fn(d.x_phys)(out)
        (out * g).sum().backward()
        res.append({n: p.grad.detach().clone() for n, p in ref.named_parameters() if p.grad is not None})
    g32, g64 = res
    scale = max(g.abs().max().item() for n, g in g64.items() if "lin_key.bias" not in n)
    floor = {n: (g32[n].double() - g).abs().max().item() / max(g.abs().max().item(), 1e-3 * scale, 1e-300)
             for n, g in g64.items()}
    return g64, floor, scale


@pytest.mark.parametrize("route", ["euler_one_launch", "rk4_one_launch", "stream", "learnable_temp"])
def test_one_step_matches_autograd_through_the_oracle(route):
    md, B, over, extra, check = ROUTES[route]
    opt, ds, data, state, extra = _case(route)
    if route != "learnable_temp":
        data = synth.make_batch((20, 20), 5, seed=3)
        opt = synth.default_opt((20, 20), num_layers=3, **over)
        ds = synth.SyntheticDataset(2, (20, 20))
        torch.manual_seed(42)
        state = copy.deepcopy(gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict())
    model, tr = _trainer(ds, opt, state, **extra)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert check(tr, s)
    x = tr.forward(sid)
    _, g = _smooth_grad_fn(data.x_phys.cuda())(x)
    tr._load_cotangent(s, g)
    with torch.cuda.stream(tr.stream):
        tr._issue(s, tr.stream.cuda_stream, with_optimizer=False)
    tr.synchronize()
    g64, floor, scale = _oracle_grads(ds, opt, data, state)
    util.check_grads_conditioned(grads_of(model), g64, floor, scale, tol=1e-4)


def _module_loop(ds, opt, state, batches, K):
    """model(data) -> grad_fn -> (x * g).sum().backward() -> torch.optim.Adam: the reference's modular loop body."""
    m = cuda_model(ds, opt, state)
    m.train()
    optim = torch.optim.Adam(m.parameters(), lr=LR)
    losses = []
    for k in range(K):
        data = batches[k % len(batches)]
        optim.zero_grad(set_to_none=True)
        out = m(data)
        loss, g = _smooth_grad_fn(data.x_phys.cuda())(out)
        (out * g.reshape(out.shape)).sum().backward()
        optim.step()
        losses.append(float(loss.item()))
    return {n: p.detach().cpu().clone() for n, p in m.named_parameters()}, losses


def _compare_params(got, want, tol=2e-3):
    assert sorted(got) == sorted(want)
    names = [n for n in want if "lin_key.bias" not in n]
    scale = max(want[n].abs().max().item() for n in names)
    worst = max((got[n] - want[n]).abs().max().item() for n in names) / scale
    print(f"max |trainer - module| / max |param| = {worst:.3e}")
    assert worst <= tol


@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("route", ["euler_one_launch", "rk4_one_launch", "glob_features", "learnable_temp"])
def test_adam_steps_match_the_module_loop(route, use_graph):
    K = 10
    opt, ds, data, state, extra = _case(route)
    batches = [data, synth.make_batch(ROUTES[route][0], ROUTES[route][1], seed=11)]
    want, want_losses = _module_loop(ds, dict(opt, loss_type="modular"), state, batches, K)
    model, tr = _trainer(ds, opt, state, use_graph=use_graph, **extra)
    losses = []
    for k in range(K):
        loss = tr.train_batch(batches[k % 2], ring=2, grad_fn=_smooth_grad_fn(batches[k % 2].x_phys.cuda()))
        losses.append(float(loss.item()))
    tr.synchronize()
    assert int(tr.step_count.item()) == K
    _compare_params({n: p.detach().cpu() for n, p in model.named_parameters()}, want)
    assert max(abs(a - b) / abs(b) for a, b in zip(losses, want_losses)) <= 1e-3


# 4 ------------------------------------------------------------------------------------------------------------------
def test_burgers_preset_through_train_batch():
    """The reference's Burgers preset (GRAND conv, 1-D meshes of 21 nodes, loss_type='modular')."""
    K, md, B = 10, (21,), 64
    opt = synth.burgers_opt(md)
    assert opt["loss_type"] == "modular"
    ds = synth.SyntheticDataset(1, md)
    batches = [synth.make_batch(md, B, seed=k, burgers=True) for k in range(2)]
    torch.manual_seed(42)
    state = copy.deepcopy(gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict())
    want, _ = _module_loop(ds, opt, state, batches, K)
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, lr=LR)
    assert tr.cot
    for k in range(K):
        tr.train_batch(batches[k % 2], ring=2, grad_fn=_smooth_grad_fn(batches[k % 2].x_phys.cuda()))
    tr.synchronize()
    assert all(tr._one_launch(s) for s in tr.slots)
    _compare_params({n: p.detach().cpu() for n, p in model.named_parameters()}, want)


# 5 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("route", ["euler_one_launch", "cluster", "learnable_temp", "gnn_normalize"])
def test_graph_replay_equals_eager_and_runs_repeat(route):
    opt, ds, data, state, extra = _case(route)
    res = []
    for use_graph in (False, True, True):
        _, tr = _trainer(ds, opt, state, use_graph=use_graph, **extra)
        sid = tr.add_batch(data)
        grad_fn = _smooth_grad_fn(data.x_phys.cuda())
        xs = []
        for _ in range(STEPS):
            x = tr.forward(sid)
            xs.append(x.clone())
            tr.step(sid, cotangent=grad_fn(x)[1])
        tr.synchronize()
        res.append((_state(tr), xs, tr.slots[sid].loss.clone()))
        tr.close()
    for other in res[1:]:
        for a, b in zip(res[0][0], other[0]):
            assert torch.equal(a, b)
        assert all(torch.equal(a, b) for a, b in zip(res[0][1], other[1]))
        assert torch.equal(res[0][2], other[2])


def test_host_cotangent_equals_device_cotangent():
    opt, ds, data, state, extra = _case("euler_one_launch")
    res = []
    for host in (False, True):
        _, tr = _trainer(ds, opt, state, **extra)
        sid = tr.add_batch(data)
        grad_fn = _smooth_grad_fn(data.x_phys.cuda())
        for _ in range(3):
            g = grad_fn(tr.forward(sid))[1]
            tr.step(sid, cotangent=g.cpu().pin_memory() if host else g)
        tr.synchronize()
        res.append(_state(tr))
    assert all(torch.equal(a, b) for a, b in zip(*res))


# 6 ------------------------------------------------------------------------------------------------------------------
def test_loopback_slot_takes_the_peer_route():
    """A cotangent slot keeps the in-kernel peer all-reduce; its local gradient (the step stopped before the exchange)
    is the loss_fn='l1' slot's bit for bit when fed that slot's cotangent, scaled for the global batch."""
    opt, ds, data, state, _ = _case("euler_one_launch")
    grads = []
    for loss_fn in ("l1", None):
        _, tr = _trainer(ds, opt, state, loss_fn=loss_fn, gad_peer_loopback=(2, 1))
        sid = tr.add_batch(data)
        s = tr.slots[sid]
        assert s.peer_route and tr._one_launch(s) and s.count_global == 2 * s.N * tr.dim
        if loss_fn is None:
            x = tr.forward(sid)
            tr._load_cotangent(s, _mesh_cotangent(x, data.x_phys.cuda().reshape(x.shape), "l1",
                                                  dp.local_grad_scale(s.N * tr.dim, s.count_global)))
        with torch.cuda.stream(tr.stream):
            tr._issue(s, tr.stream.cuda_stream, with_optimizer=False)
        tr.stream.synchronize()
        grads.append(tr.gflat.detach().clone())
        tr.close()
    assert torch.equal(grads[0], grads[1])


@pytest.mark.timeout(300)
def test_two_gpus_match_one_gpu_on_the_union_batch(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, B, steps = 2, 3, 6
    out = tmp_path / "dp_modular.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29547",
           os.path.join(ROOT, "tests", "dp_modular_worker.py"), str(out), str(steps), str(B)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads(out.read_text())
    md = (12, 12)
    for key, extra in (("peer", {}), ("nccl", {"gad_peer_allreduce": False})):
        got = res[key]
        assert got["ranks_equal"] and got["selfcheck"]["ranks_equal"]
        assert got["peer_route"] == (key == "peer")
        opt = synth.default_opt(md, lr=1e-2, loss_type="modular")
        torch.manual_seed(42)
        model = cuda_model(synth.SyntheticDataset(2, md), opt, gad_store_alpha=False)
        tr = DeformerTrainer(model, lr=1e-2)
        data = [synth.make_batch(md, world * B, seed=7, first_mesh_id=k * world * B) for k in range(2)]
        sids = [tr.add_batch(d) for d in data]
        for k in range(steps):
            x = tr.forward(sids[k % 2])
            tr.step(sids[k % 2], cotangent=_smooth_grad_fn(data[k % 2].x_phys.cuda())(x)[1])
        tr.synchronize()
        want = tr.flat.cpu()
        flat = torch.tensor(got["flat"])
        live = torch.ones(want.numel(), dtype=torch.bool)
        o = (tr.bk.data_ptr() - tr.flat.data_ptr()) // 4
        live[o:o + tr.bk.numel()] = False            # lin_key.bias: analytically zero gradient
        err = (flat - want)[live].abs().max().item() / want[live].abs().max().item()
        assert err <= 2e-3, (key, err)


# 7 ------------------------------------------------------------------------------------------------------------------
def test_refusals():
    opt, ds, data, state, _ = _case("euler_one_launch")
    _, tr = _trainer(ds, opt, state)
    sid = tr.add_batch(data)
    sid2 = tr.add_batch(synth.make_batch((30, 30), 8, seed=6))
    x = tr.forward(sid)
    with pytest.raises(ValueError, match="needs the cotangent"):
        tr.step(sid)
    for bad in (torch.zeros(x.shape[0], 3, device="cuda"), torch.zeros(x.shape[0], device="cuda"),
                torch.zeros(x.shape, dtype=torch.float64, device="cuda"), x.tolist()):
        with pytest.raises(ValueError, match="float32 tensor of shape"):
            tr.step(sid, cotangent=bad)
    with pytest.raises(ValueError, match="pinned"):
        tr.step(sid, cotangent=torch.zeros(x.shape))
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="trainer runs on"):
            tr.step(sid, cotangent=torch.zeros(x.shape, device="cuda:1"))
    for call in (lambda: tr.run_epoch([sid, sid2]), lambda: tr.capture_epoch([sid, sid2]),
                 lambda: tr.run_from_host([tr.pack_host(sid, data), tr.pack_host(sid2, data)], 2),
                 lambda: tr.step_from_host(sid, data)):
        with pytest.raises(ValueError, match="loss_type='modular'"):
            call()
    with pytest.raises(ValueError, match="cotangent mode"):
        tr.train_batch(data)
    assert int(tr.step_count.item()) == 0
    _, ref = _trainer(ds, opt, state, loss_fn="l1")
    rid = ref.add_batch(data)
    with pytest.raises(ValueError, match="cotangent mode"):
        ref.forward(rid)
    with pytest.raises(ValueError, match="loss_type='modular'"):
        ref.step(rid, cotangent=x)
    with pytest.raises(ValueError, match="loss_type='modular' only"):
        ref.train_batch(data, grad_fn=_smooth_grad_fn(data.x_phys.cuda()))


def test_c_abi_takes_loss_kind_2_and_rejects_3():
    lib, P = _lib.load(), _lib.ptr
    opt, ds, data, state, _ = _case("euler_one_launch")
    _, tr = _trainer(ds, opt, state)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    for kind, rc in ((2, 0), (3, 1)):
        d = tr._train_desc(s, 1)
        assert d.loss_kind == 2 and d.grad_scale == 1.0 and d.loss_scale == 1.0
        d.loss_kind = kind
        for fn in ("gad_train_step_ell", "gad_train_step_ell_rk4", "gad_train_step_cluster"):
            if kind == 2 and fn != "gad_train_step_ell":
                continue          # a mesh-resident Euler slot: the other two kernels do not take its descriptor
            args = (ctypes.byref(d), 2, None) if fn == "gad_train_step_cluster" else (ctypes.byref(d), None)
            assert getattr(lib, fn)(*args) == rc, fn
            if rc:
                assert "unknown loss kind 3" in lib.gad_last_error().decode()
        torch.cuda.synchronize()
        n = s.N * tr.dim
        assert lib.gad_mesh_loss(P(s.x_phys), P(s.target), n, kind, 1.0, P(s.loss), P(s.g_out), P(s.loss_ws), None) == rc
        torch.cuda.synchronize()
        if kind == 2:        # loss = <out, c> (a sum), g_out = grad_scale * c
            assert torch.equal(s.g_out, s.target)
            want = (s.x_phys.double() * s.target.double()).sum().item()
            assert abs(s.loss.item() - want) <= 1e-5 * max(abs(want), 1e-30) + 1e-7
    assert lib.gad_mesh_loss(P(s.x_phys), P(s.target), s.N * tr.dim, 3, 1.0, P(s.loss), None, P(s.loss_ws), None) == 1
    assert "gad_mesh_loss" in lib.gad_last_error().decode()
