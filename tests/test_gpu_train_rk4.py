"""DeformerTrainer on ode_method='rk4': the one-launch step (csrc/ell_kernels.cuh: k_ell_train<..., GAD_METHOD_RK4>,
gad_train_step_ell_rk4) on tiles that fit its nine rows per node, the launch chain (forward, mesh loss, RK4 backward,
weight gradients, Adam) everywhere else.

Bars are the project's: loss 1e-5 relative and parameter gradients 1e-4 against autograd through the oracle's RK4 in
fp64 (widened to 4 x the fp32 oracle's own deviation where that is larger, gad_testutil.fp64_grads_and_noise_floor);
the module path and the separate-kernel route within the bars of test_gpu_ell; Adam within those of
test_gpu_train_adam; determinism, topology forms and loop shapes bit for bit.
"""
import copy

import pytest
import torch
import torch.nn.functional as F

from g_adaptivity_b200 import synth
from g_adaptivity_b200.trainer import DeformerTrainer
from test_gpu_parity import cuda_model, grads_of, oracle_model
from test_gpu_peer_loopback import _local_gradient, _ordered_sum, _trainer

import gad_testutil as util

pytestmark = pytest.mark.gpu

RK4 = {"ode_method": "rk4"}


def _case(mesh_dims, B, seed=0, burgers=False, **over):
    over = dict(RK4, **over)
    opt = synth.burgers_opt(mesh_dims, **over) if burgers else synth.default_opt(mesh_dims, **over)
    ds = synth.SyntheticDataset(len(mesh_dims), mesh_dims)
    data = synth.make_batch(mesh_dims, B, seed=seed, burgers=burgers)
    torch.manual_seed(42)
    state = copy.deepcopy(oracle_model(ds, opt).state_dict())
    return opt, ds, data, state


def _oracle_loss_and_grads(ds, opt, data, state, loss_fn):
    """Loss and parameter gradients of the oracle's RK4 in fp64, and the fp32 oracle's deviations from them (the loss
    bar widens to 4 x the fp32 oracle's own deviation where that is larger, as the gradient bar does: on 1-D meshes of
    thousands of nodes the loss is a mean of |x - target| ~ 1e-5 over coordinates ~ 1)."""
    lossf = F.l1_loss if loss_fn == "l1" else F.mse_loss
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
        loss = lossf(out, d.x_phys.reshape(out.shape))
        loss.backward()
        res.append((loss.item(), {n: p.grad.detach().clone() for n, p in ref.named_parameters() if p.grad is not None}))
    (l32, g32), (l64, g64) = res
    scale = max(g.abs().max().item() for n, g in g64.items() if "lin_key.bias" not in n)
    floor = {n: (g32[n].double() - g).abs().max().item() / max(g.abs().max().item(), 1e-3 * scale, 1e-300)
             for n, g in g64.items()}
    loss_tol = max(1e-5, 4.0 * abs(l32 - l64) / abs(l64))
    return l64, loss_tol, g64, floor, scale


def _step_without_optimizer(tr, sid):
    with torch.cuda.stream(tr.stream):
        tr._issue(tr.slots[sid], tr.stream.cuda_stream, with_optimizer=False)
    tr.synchronize()
    return tr.slots[sid].loss.item()


# 1 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("loss_fn", ["l1", "mse"])
@pytest.mark.parametrize("mesh_dims,B,burgers,over", [
    ((20, 20), 7, False, {"num_layers": 3}),
    ((30, 30), 5, False, {"num_layers": 2, "share_conv": False}),
    ((12, 12), 9, False, {"num_layers": 4, "self_loops": True, "time_step": 0.3}),
    ((40,), 33, True, {"num_layers": 3}),
])
def test_one_launch_step_matches_autograd_through_the_oracle(mesh_dims, B, burgers, over, loss_fn):
    opt, ds, data, state = _case(mesh_dims, B, seed=3, burgers=burgers, **over)
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, loss_fn=loss_fn, use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert s.rk4_fused and tr._one_launch(s)
    loss = _step_without_optimizer(tr, sid)
    l64, loss_tol, g64, floor, scale = _oracle_loss_and_grads(ds, opt, data, state, loss_fn)
    assert abs(loss - l64) <= loss_tol * abs(l64), (loss, l64, loss_tol)
    util.check_grads_conditioned(grads_of(model), g64, floor, scale, tol=1e-4)


# 2 ------------------------------------------------------------------------------------------------------------------
def test_one_launch_step_equals_the_module_path():
    """Same parameters, same batch: x_phys of the one-launch step is GNN.forward's bit for bit (same forward
    expressions on the same inputs); the gradient is F.l1_loss(model(data), target).backward()'s within 1e-5 of its
    largest entry (the per-tile partials are reduced in another order)."""
    opt, ds, data, state = _case((30, 30), 24, seed=6)
    m = cuda_model(ds, opt, state)
    m.train()
    out = m(data)
    F.l1_loss(out, data.x_phys.cuda()).backward()
    want = grads_of(m)
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(data)
    assert tr.slots[sid].rk4_fused
    _step_without_optimizer(tr, sid)
    assert torch.equal(tr.slots[sid].x_phys, out.detach())
    got = grads_of(model)
    scale = max(g.abs().max().item() for g in want.values())
    worst = max((got[n] - g).abs().max().item() for n, g in want.items())
    print(f"module path vs one launch: x_phys bit-identical; gradient max |diff| / scale = {worst / scale:.3e}, "
          f"bit-identical: {all(torch.equal(got[n], g) for n, g in want.items())}")
    assert worst <= 1e-5 * scale


# 3 ------------------------------------------------------------------------------------------------------------------
def test_one_launch_step_equals_the_launch_chain():
    opt, ds, data, state = _case((30, 30), 24, seed=6)
    res = []
    for no_fused in (False, True):
        model = cuda_model(ds, opt, state, gad_no_fused_train=no_fused, gad_store_alpha=False)
        tr = DeformerTrainer(model, use_cuda_graph=False)
        sid = tr.add_batch(data)
        assert tr.slots[sid].rk4_fused and tr._fused_ell(tr.slots[sid]) != no_fused
        loss = _step_without_optimizer(tr, sid)
        res.append((loss, tr.gflat.clone().cpu()))
    assert abs(res[0][0] - res[1][0]) <= 1e-6 * abs(res[1][0])
    assert (res[0][1] - res[1][1]).abs().max().item() <= 1e-5 * res[1][1].abs().max().item()
    res = []
    for no_fused in (False, True):
        model = cuda_model(ds, opt, state, gad_no_fused_train=no_fused, gad_store_alpha=False)
        tr = DeformerTrainer(model, lr=3e-3)
        sid = tr.add_batch(data)
        for _ in range(6):
            tr.step(sid)
        tr.synchronize()
        res.append((tr.flat.clone().cpu(), tr.slots[sid].loss.item(), int(tr.step_count.item())))
    assert res[0][2] == res[1][2] == 6
    assert abs(res[0][1] - res[1][1]) <= 2e-5 * abs(res[1][1])
    assert (res[0][0] - res[1][0]).abs().max().item() <= 2e-5 * res[1][0].abs().max().item()


# 4 ------------------------------------------------------------------------------------------------------------------
MD, K, LR = (30, 30), 10, 1e-2


def _flat_views(model):
    c = model.conv_layers[0]
    return [c.lin_query.weight, c.lin_query.bias, c.lin_key.weight, c.lin_key.bias]


@pytest.fixture(scope="module")
def adam_case():
    opt = synth.default_opt(MD, lr=LR, **RK4)
    ds = synth.SyntheticDataset(2, MD)
    batches = [synth.make_batch(MD, 64, seed=31, first_mesh_id=r * 64) for r in range(2)]
    torch.manual_seed(42)
    state = copy.deepcopy(oracle_model(ds, opt).state_dict())
    m = cuda_model(ds, opt, state)                           # the module path trained by torch.optim.Adam
    m.train()
    optim = torch.optim.Adam(m.parameters(), lr=LR)
    losses = []
    for k in range(K):
        data = batches[k % 2]
        optim.zero_grad(set_to_none=True)
        loss = F.l1_loss(m(data), data.x_phys.cuda())
        loss.backward()
        optim.step()
        losses.append(float(loss.item()))
    want = torch.cat([v.detach().flatten() for v in _flat_views(m)]).cpu()
    return opt, ds, batches, state, want, losses


@pytest.mark.parametrize("mode", ["eager", "graph", "epoch"])
def test_k_steps_match_the_module_path_trained_by_torch_adam(adam_case, mode):
    opt, ds, batches, state, want, ref_losses = adam_case
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=(mode != "eager"))
    sids = [tr.add_batch(b) for b in batches]
    assert tr._one_launch(tr.slots[0]) and tr.slots[0].rk4_fused
    losses = []
    if mode == "epoch":
        for _ in range(K // 2):
            tr.run_epoch(sids)
            tr.synchronize()
            losses += [float(tr.slots[s].loss.item()) for s in sids]
    else:
        for k in range(K):
            l = tr.step(sids[k % 2])
            tr.synchronize()
            losses.append(float(l.item()))
    assert int(tr.step_count.item()) == K
    got = tr.flat.detach().cpu()
    n = got.numel()
    live = torch.ones(n, dtype=torch.bool)
    live[n - _flat_views(model)[3].numel():] = False        # lin_key.bias: gradient analytically zero
    assert abs(losses[0] - ref_losses[0]) <= 1e-5 * abs(ref_losses[0])
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 2e-3 * abs(b), (losses, ref_losses)
    assert losses[-1] < losses[0]
    err = (got - want)[live].abs().max().item() / want[live].abs().max().item()
    assert err <= 2e-3, err
    assert torch.equal(got[~live], state["conv_layers.0.lin_key.bias"].flatten())


@pytest.mark.parametrize("mode,wd,over", [
    ("eager", 0.0, {}),
    ("graph", 0.0, {}),
    ("epoch", 0.0, {}),
    ("graph", 1e-2, {}),
    ("graph", 0.0, {"share_conv": False}),
])
def test_adam_arithmetic_equals_torch_optim_adam_on_the_same_gradients(mode, wd, over):
    opt = synth.default_opt(MD, lr=LR, decay=wd, **RK4, **over)
    ds = synth.SyntheticDataset(2, MD)
    batches = [synth.make_batch(MD, 16, seed=32, first_mesh_id=r * 16) for r in range(2)]
    torch.manual_seed(42)
    state = oracle_model(ds, opt).state_dict()
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=(mode != "eager"))
    assert tr.wd == wd
    sids = [tr.add_batch(b) for b in batches]
    assert tr._one_launch(tr.slots[0])
    shadow = torch.nn.Parameter(tr.flat.detach().cpu().clone())
    optim = torch.optim.Adam([shadow], lr=LR, weight_decay=wd)
    scale = shadow.detach().abs().max().item()
    for k in range(K):
        if mode == "epoch":
            tr.run_epoch([sids[k % 2]])
        else:
            tr.step(sids[k % 2])
        tr.synchronize()
        shadow.grad = tr.gflat.detach().cpu().clone()
        optim.step()
        err = (tr.flat.detach().cpu() - shadow.detach()).abs().max().item() / scale
        assert err <= 1e-6, err
    assert int(tr.step_count.item()) == K


# 5 ------------------------------------------------------------------------------------------------------------------
def _replayed(opt, ds, data, state, steps, loss_fn=None, **extra):
    model = cuda_model(ds, opt, state, gad_store_alpha=False, **extra)
    tr = DeformerTrainer(model, lr=1e-2, loss_fn=loss_fn)
    sid = tr.add_batch(data)
    losses = []
    for _ in range(steps):
        loss = tr.step(sid)
        with torch.cuda.stream(tr.stream):
            losses.append(loss.clone())
    tr.synchronize()
    return tr, sid, [float(x.item()) for x in losses], tr.flat.clone().cpu()


def test_graph_replay_is_deterministic_and_trains():
    opt, ds, data, state = _case((30, 30), 32, seed=8)
    a = _replayed(opt, ds, data, state, 12)
    b = _replayed(opt, ds, data, state, 12)
    assert a[0].slots[a[1]].rk4_fused
    assert a[2] == b[2] and torch.equal(a[3], b[3])
    assert a[2][-1] < a[2][0]


# 6 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mesh_dims,B,burgers,over", [
    ((50, 50), 2, False, {"num_layers": 3}),      # 2500-node tiles: nine rows per node do not fit a CTA
    ((64, 64), 1, False, {"num_layers": 2}),      # beyond one CTA
    ((3000,), 2, True, {"num_layers": 3}),
])
def test_launch_chain_shapes(mesh_dims, B, burgers, over):
    opt, ds, data, state = _case(mesh_dims, B, seed=3, burgers=burgers, **over)
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, loss_fn="l1", use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert not tr._one_launch(s) and not s.rk4_fused
    loss = _step_without_optimizer(tr, sid)
    l64, loss_tol, g64, floor, scale = _oracle_loss_and_grads(ds, opt, data, state, "l1")
    assert abs(loss - l64) <= loss_tol * abs(l64), (loss, l64, loss_tol)
    util.check_grads_conditioned(grads_of(model), g64, floor, scale, tol=1e-4)
    a = _replayed(opt, ds, data, state, 4, loss_fn="l1")
    b = _replayed(opt, ds, data, state, 4, loss_fn="l1")
    assert a[2] == b[2] and torch.equal(a[3], b[3])


# 7 ------------------------------------------------------------------------------------------------------------------
def test_shared_topology_trains_like_the_general_graph():
    opt, ds, data, state = _case((20, 20), 12, seed=13)
    outs = []
    for shared in (False, True):
        tr, sid, losses, flat = _replayed(opt, ds, data, state, 5, gad_shared_topology=shared)
        assert tr.slots[sid].graph.uniform == shared and tr.slots[sid].rk4_fused
        outs.append((losses, flat))
    assert outs[0][0] == outs[1][0] and torch.equal(outs[0][1], outs[1][1])


# 8 ------------------------------------------------------------------------------------------------------------------
def test_train_batch_and_run_from_host_equal_resident_steps():
    opt, ds, _, state = _case((20, 20), 12, seed=3)
    fresh = [synth.make_batch((20, 20), 12, seed=50 + k) for k in range(5)]
    for b in fresh:
        b.pin_memory()
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, lr=1e-2)
    got = []
    for b in fresh:
        loss = tr.train_batch(b)
        tr.synchronize()
        got.append(float(loss.item()))
    model2 = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr2 = DeformerTrainer(model2, lr=1e-2)
    sids = [tr2.add_batch(b) for b in fresh]
    want = []
    for sid in sids:
        loss = tr2.step(sid)
        tr2.synchronize()
        want.append(float(loss.item()))
    assert got == want and torch.equal(tr.flat, tr2.flat)

    batches = fresh[:2]
    outs = []
    for mode in ("resident", "packed_native"):
        model = cuda_model(ds, opt, state, gad_store_alpha=False)
        tr = DeformerTrainer(model, lr=1e-2)
        sids = [tr.add_batch(b) for b in batches]
        if mode == "resident":
            losses = []
            for k in range(6):
                l = tr.step(sids[k % 2])
                with torch.cuda.stream(tr.stream):
                    losses.append(l.clone())
            tr.synchronize()
            losses = torch.stack([x.cpu() for x in losses]).reshape(-1)
        else:
            src = [tr.pack_host(sid, b) for sid, b in zip(sids, batches)]
            losses = tr.run_from_host(src, 6, native=True).clone()
        outs.append((losses, tr.flat.clone().cpu()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


# 9 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world,rank", [(2, 1), (8, 5)])
def test_in_kernel_allreduce_is_the_rank_ordered_sum_and_adam_consumes_it(world, rank):
    tr, sid = _trainer(world, rank, ode_method="rk4")
    assert tr.slots[sid].rk4_fused
    shadow = torch.nn.Parameter(tr.flat.detach().cpu().clone())
    optim = torch.optim.Adam([shadow], lr=1e-2)
    gen = torch.Generator().manual_seed(100 + world * 16 + rank)
    for seq in (1, 2, 3):
        g_own = _local_gradient(tr, sid)
        parts = []
        for r in range(world):
            if r == rank:
                parts.append(g_own)
                continue
            g_r = (g_own.cpu() * (0.5 + torch.rand(g_own.numel(), generator=gen))).to(g_own.device)
            tr.peer.peer_words(seq, r, g_r)
            parts.append(g_r)
        want = _ordered_sum(parts)
        tr.step(sid)
        tr.synchronize()
        assert int(tr.peer.seq[0].item()) == seq and int(tr.peer.seq[1].item()) == 0
        assert torch.equal(tr.gflat, want)
        shadow.grad = want.cpu().clone()
        optim.step()
        err = (tr.flat.detach().cpu() - shadow.detach()).abs().max().item() / shadow.detach().abs().max().item()
        assert err <= 1e-6, err


# 10 -----------------------------------------------------------------------------------------------------------------
def test_learn_step_is_refused():
    opt = synth.default_opt((10, 10), learn_step=True, **RK4)
    model = cuda_model(synth.SyntheticDataset(2, (10, 10)), opt)
    with pytest.raises(NotImplementedError):
        DeformerTrainer(model)
