"""DeformerTrainer with gnn_normalize=True and softmax_temp_type='learnable_a'.

gnn_normalize (src/GNN.py:231-237: f / torch.max(f), uu / torch.max(uu) over the batch) keeps every route of the
trainer: the step starts with gad_batch_max over the slot's resident f / uu, whose results are the f_scale / uu_scale
the kernels divide by.  The learnable temperature (one trainable sm_temp_a per weight set) trains through the chain of
library kernels: gad_temp_fold (Mu / temp) before the deformer forward, gad_temp_fold_bwd (the temperature's gradient
and the cotangent of the base weights) after its backward.

On the chain the trainer runs the kernels GNN.forward + autograd run, so on identical parameters the folded weights,
x_phys and every gradient equal the module path's bit for bit -- except the temperature's gradient, which the module
sums with torch (compared within 1e-6 of its largest entry).  A normalised slot on the one-launch kernel k_ell_train is
compared at the bars of the other one-launch tests (coordinates and loss 1e-5, gradients 1e-4)."""
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
from test_gpu_parity import check_grads, cuda_model, grads_of
from test_gpu_train_pde_loss import _case as _pde_case

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NORM = dict(gnn_normalize=True)
TEMP = dict(softmax_temp_type="learnable_a")
BOTH = dict(gnn_normalize=True, softmax_temp_type="learnable_a")


def _scale_features(data, B, first_mesh_id=0):
    """f and uu of mesh j times (1 + j % 3) and (2 - 0.5 * (j % 2)): batches and shards with different maxima."""
    n = data.f_tensor.numel() // B
    j = torch.arange(first_mesh_id, first_mesh_id + B, dtype=torch.float32).repeat_interleave(n)
    data.f_tensor = data.f_tensor * (1.0 + j % 3)
    data.uu_tensor = data.uu_tensor * (2.0 - 0.5 * (j % 2))
    return data


def _case(md, B, seed=9, first_mesh_id=0, **over):
    """opt, dataset, batch and initial parameters of a mesh-loss case; a pde case when over has loss_type='pde_loss'."""
    if over.get("loss_type") == "pde_loss":
        over = dict(over)
        del over["loss_type"]
        opt, ds, data, state = _pde_case(md, B, seed=seed, **over)
        return opt, ds, _scale_features(data, B), state
    opt = synth.default_opt(md, **over)
    ds = synth.SyntheticDataset(len(md), md)
    data = _scale_features(synth.make_batch(md, B, seed=seed, first_mesh_id=first_mesh_id), B, first_mesh_id)
    torch.manual_seed(42)
    state = copy.deepcopy(gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict())
    return opt, ds, data, state


def _batches(opt, md, B, n, seed=31):
    pde = opt["loss_type"] == "pde_loss"
    Q = opt["eval_quad_points"]
    return [_scale_features(synth.make_batch(md, B, seed=seed, first_mesh_id=r * B, eval_quad_points=Q,
                                             with_u_true_fine=pde and len(md) == 2), B, r * B) for r in range(n)]


def _step_without_optimizer(tr, sid):
    with torch.cuda.stream(tr.stream):
        tr._issue(tr.slots[sid], tr.stream.cuda_stream, with_optimizer=False)
    tr.synchronize()
    return tr.slots[sid].loss.item()


def _module_loss(opt, m, data):
    """GNN.forward with autograd and the loss the trainer takes: (x_phys, loss)."""
    m.train()
    out = m(data)
    if opt["loss_type"] == "pde_loss":
        _, x_phys, sol = out
        return x_phys, F.mse_loss(sol, data.u_true_fine_tensor.cuda())
    lossf = F.l1_loss if opt.get("loss_fn", "l1") == "l1" else F.mse_loss
    return out, lossf(out, data.x_phys.cuda().reshape(out.shape))


def _trainer(ds, opt, state, graph=False, lr=None, **extra):
    model = cuda_model(ds, opt, state, gad_store_alpha=False, **extra)
    loss_fn = None if opt["loss_type"] == "pde_loss" else opt.get("loss_fn", "l1")
    return model, DeformerTrainer(model, lr=lr, loss_fn=loss_fn, use_cuda_graph=graph)


# 1 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["normalize_6x6", "temp_learnable_a_7x7", "temp_learnable_a_noshare_6x6"])
def test_one_step_matches_the_reference_fixture(name):
    """Bars of test_gpu_parity.py::test_deformer_matches_reference_fixture: coordinates and loss 1e-5, gradients 1e-4
    (sm_temp_a included)."""
    fx = util.load_golden(name)
    opt = util.fixture_opt(fx)
    data = util.fixture_batch(fx)
    model = cuda_model(util.fixture_dataset(fx), opt, fx["state_dict"], gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert s.norm == bool(opt["gnn_normalize"]) and s.temp == (opt.get("softmax_temp_type") == "learnable_a")
    assert tr._one_launch(s) == (not s.temp)
    loss = _step_without_optimizer(tr, sid)
    assert util.rel_err(s.x_phys.reshape(fx["x_phys"].shape), fx["x_phys"]) <= 1e-5
    assert abs(loss - fx["loss"]) <= 1e-5 * abs(fx["loss"]), (loss, fx["loss"])
    got = grads_of(model)
    assert any("sm_temp_a" in n for n in got) == s.temp
    check_grads(got, fx["grads"])


# 2 ------------------------------------------------------------------------------------------------------------------
LINK_ROWS = [
    ((7, 7), 3, dict(TEMP)),
    ((7, 7), 3, dict(TEMP, ode_method="rk4")),
    ((7, 7), 3, dict(TEMP, share_conv=False, num_layers=3, loss_fn="mse")),
    ((7, 7), 3, dict(BOTH, learn_step=True)),
    ((30, 30), 16, dict(BOTH, share_conv=False, ode_method="rk4")),
    ((200,), 16, dict(BOTH)),
    ((7, 7), 3, dict(BOTH, loss_type="pde_loss", Q=13, K=9)),
    ((200,), 16, dict(BOTH, loss_type="pde_loss", share_conv=False)),
    ((7, 7), 3, dict(NORM, loss_type="pde_loss", Q=13, K=9, ode_method="rk4")),
]


def _row_id(r):
    md, B, over = r
    extra = "-".join(f"{k}={v}" for k, v in over.items() if k not in ("Q", "K"))
    return "x".join(map(str, md)) + f"-B{B}-" + extra


@pytest.mark.parametrize("row", LINK_ROWS, ids=[_row_id(r) for r in LINK_ROWS])
def test_chain_matches_the_module_path_link_by_link(row):
    md, B, over = row
    opt, ds, data, state = _case(md, B, **over)
    model, tr = _trainer(ds, opt, state)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert s.chain and not tr._one_launch(s)
    got_loss = _step_without_optimizer(tr, sid)
    m = cuda_model(ds, opt, state, gad_store_alpha=False)
    assert torch.equal(s.graph.ell_tile_ptr, m._graph(data, tr.dev, True).ell_tile_ptr)
    x_phys, loss = _module_loss(opt, m, data)
    if s.norm:
        assert s.f_scale.item() == data.f_tensor.max().item() and s.uu_scale.item() == data.uu_tensor.max().item()
    if s.temp:
        convs = [m.conv_layers[0]] if opt["share_conv"] else list(m.conv_layers)
        temp = torch.cat([c.sm_temp_a.detach().reshape(1) for c in convs])
        assert torch.equal(tr.Mu_eff, m._folded_weights(tr.dev) * (1.0 / temp.reshape(-1, 1)))
    assert torch.equal(s.x_phys.reshape(-1), x_phys.detach().reshape(-1))
    assert abs(got_loss - loss.item()) <= 1e-6 * abs(loss.item()), (got_loss, loss.item())
    # the module's backward of the trainer's own cotangent of x_phys (the 2-D FEM backward's fp64 atomics leave the
    # last bit of that cotangent open, test_gpu_train_pde_loss.py)
    m.zero_grad(set_to_none=True)
    x_phys.backward(s.g_out.reshape(x_phys.shape))
    want = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in model.named_parameters() if n in want}
    assert sorted(got) == sorted(want) and any("sm_temp_a" in n for n in want) == s.temp
    for n in want:
        if "sm_temp_a" in n:
            continue
        assert torch.equal(got[n], want[n]), n
    if s.temp:
        gt = torch.cat([got[n].reshape(1) for n in sorted(want) if "sm_temp_a" in n])
        wt = torch.cat([want[n].reshape(1) for n in sorted(want) if "sm_temp_a" in n])
        assert (gt - wt).abs().max().item() <= 1e-6 * wt.abs().max().item(), (gt, wt)


@pytest.mark.parametrize("md,B,over", [((6, 6), 4, dict(NORM)), ((30, 30), 64, dict(NORM, loss_fn="mse")),
                                       ((30, 30), 64, dict(NORM, ode_method="rk4", share_conv=False)),
                                       ((200,), 64, dict(NORM, learn_step=True))])
def test_normalised_one_launch_step_matches_the_module_path(md, B, over):
    opt, ds, data, state = _case(md, B, **over)
    model, tr = _trainer(ds, opt, state)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert s.norm and tr._one_launch(s)
    got_loss = _step_without_optimizer(tr, sid)
    m = cuda_model(ds, opt, state, gad_store_alpha=False)
    x_phys, loss = _module_loss(opt, m, data)
    loss.backward()
    assert util.rel_err(s.x_phys, x_phys.reshape(s.x_phys.shape)) <= 1e-5
    assert abs(got_loss - loss.item()) <= 1e-5 * abs(loss.item())
    check_grads(grads_of(model), grads_of(m))


# 3 ------------------------------------------------------------------------------------------------------------------
K_STEPS, LR = 10, 1e-2
ADAM_ROWS = [
    ((7, 7), 4, dict(TEMP)),
    ((7, 7), 4, dict(NORM)),
    ((7, 7), 4, dict(BOTH, ode_method="rk4", share_conv=False, num_layers=3, loss_fn="mse")),
    ((7, 7), 4, dict(NORM, ode_method="rk4", share_conv=False, num_layers=3, loss_fn="mse")),
    ((30, 30), 256, dict(TEMP, loss_fn="mse")),
    ((30, 30), 256, dict(NORM)),
    ((30, 30), 256, dict(BOTH, ode_method="rk4")),
    ((7, 7), 4, dict(BOTH, loss_type="pde_loss", Q=13, K=9)),
    ((200,), 32, dict(BOTH, loss_type="pde_loss", share_conv=False)),
]
_ADAM_REF = {}


def _module_adam(opt, ds, state, batches):
    m = cuda_model(ds, opt, state, gad_store_alpha=False)
    optim = torch.optim.Adam(m.parameters(), lr=LR)
    losses = []
    for k in range(K_STEPS):
        optim.zero_grad(set_to_none=True)
        _, loss = _module_loss(opt, m, batches[k % len(batches)])
        loss.backward()
        optim.step()
        losses.append(float(loss.item()))
    return {n: p.detach().cpu().clone() for n, p in m.named_parameters()}, losses


def _adam_case(i):
    if i not in _ADAM_REF:
        md, B, over = ADAM_ROWS[i]
        opt, ds, _, state = _case(md, B, **over)
        batches = _batches(opt, md, B, 2)
        _ADAM_REF[i] = (opt, ds, state, batches, *_module_adam(opt, ds, state, batches))
    return _ADAM_REF[i]


def _trainer_run(ds, opt, state, batches, mode):
    model, tr = _trainer(ds, opt, state, graph=mode != "eager", lr=LR)
    sids = [tr.add_batch(b) for b in batches]
    losses = []
    if mode == "epoch":
        for _ in range(K_STEPS // len(sids)):
            tr.run_epoch(sids)
            tr.synchronize()
            losses += [float(tr.slots[s].loss.item()) for s in sids]
    else:
        for k in range(K_STEPS):
            l = tr.step(sids[k % len(sids)])
            tr.synchronize()
            losses.append(float(l.item()))
    assert int(tr.step_count.item()) == K_STEPS
    return tr, {n: p.detach().cpu().clone() for n, p in model.named_parameters()}, losses


@pytest.mark.parametrize("mode", ["eager", "graph", "epoch"])
@pytest.mark.parametrize("i", range(len(ADAM_ROWS)), ids=[_row_id(r) for r in ADAM_ROWS])
def test_k_adam_steps_match_the_module_path(i, mode):
    """The project's Adam bar: 2e-3 of the largest parameter after K steps (lin_key.bias excluded: its gradient is
    analytically zero, so Adam turns rounding noise into O(lr)); torch.optim.Adam and gad_adam_step round apart."""
    opt, ds, state, batches, want, ref_losses = _adam_case(i)
    tr, got, losses = _trainer_run(ds, opt, state, batches, mode)
    s = tr.slots[0]
    assert s.chain == (s.temp or s.pde)
    assert sorted(got) == sorted(want) and any("sm_temp_a" in n for n in got) == s.temp
    names = [n for n in want if "lin_key.bias" not in n]
    scale = max(want[n].abs().max().item() for n in names)
    worst = max((got[n] - want[n]).abs().max().item() for n in names) / scale
    print(f"parameters after {K_STEPS} Adam steps: max |trainer - module| / max |param| = {worst:.3e}")
    assert worst <= 2e-3, worst
    if s.temp:      # the temperatures train (as on the module path)
        assert any(not torch.equal(got[n], state[n]) for n in names if "sm_temp_a" in n)
    assert abs(losses[0] - ref_losses[0]) <= 1e-5 * abs(ref_losses[0])
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 2e-3 * abs(b), (losses, ref_losses)


# 4 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("over", [NORM, BOTH], ids=["normalize-one-launch", "normalize-learnable_a-chain"])
def test_fresh_inputs_are_normalised_by_their_own_maxima(over):
    """lr = 0: every step runs at the initial parameters, so each step's loss must be the module's on the batch that step
    consumed.  The batches' f / uu maxima differ (by up to 3x), so a maximum left over from another batch shows."""
    md, B = (7, 7), 4
    opt, ds, _, state = _case(md, B, **over)
    fresh = _batches(opt, md, B, 4, seed=50)
    assert len({b.f_tensor.max().item() for b in fresh}) == 4 and len({b.uu_tensor.max().item() for b in fresh}) > 1
    for b in fresh:
        b.pin_memory()
    m = cuda_model(ds, opt, state, gad_store_alpha=False)
    want = [_module_loss(opt, m, b)[1].item() for b in fresh]
    tol = 1e-5 if over is NORM else 1e-6

    def check(losses, order):
        for l, k in zip(losses, order):
            assert abs(float(l) - want[k]) <= tol * abs(want[k]), (k, float(l), want[k])

    _, tr = _trainer(ds, opt, state, graph=True, lr=0.0, gad_shared_topology=True)
    got = []
    for k in range(8):
        l = tr.train_batch(fresh[k % 4], ring=2)          # one ring of two slots, refilled in turn
        tr.synchronize()
        got.append(float(l.item()))
    assert len(tr.slots) == 2
    check(got, [k % 4 for k in range(8)])
    assert tr._one_launch(tr.slots[0]) == (over is NORM)
    for native in (True, False):
        _, tr = _trainer(ds, opt, state, graph=True, lr=0.0)
        sids = [tr.add_batch(b) for b in fresh[:2]]
        src = [tr.pack_host(sids[0], b) for b in fresh] if native else fresh
        losses = tr.run_from_host(src, 8, native=native).clone()
        check(losses.tolist(), [k % 4 for k in range(8)])


# 5 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("md,over", [((7, 7), NORM), ((12, 12), BOTH), ((200,), dict(BOTH, loss_type="pde_loss"))],
                         ids=["normalize", "normalize-learnable_a", "pde-1d"])
def test_steps_are_bit_reproducible(md, over):
    """1-D for the pde loss: the 2-D FEM backward's fp64 shared-memory atomics leave the last bit open."""
    opt, ds, _, state = _case(md, 4, **over)
    batches = _batches(opt, md, 4, 2)
    runs = [_trainer_run(ds, opt, state, batches, "graph") for _ in range(2)]
    assert runs[0][2] == runs[1][2] and torch.equal(runs[0][0].flat, runs[1][0].flat)
    _, flat_e, losses_e = _trainer_run(ds, opt, state, batches, "epoch")
    assert losses_e == runs[0][2] and all(torch.equal(flat_e[n], runs[0][1][n]) for n in flat_e)


# 6 ------------------------------------------------------------------------------------------------------------------
def test_refusals():
    opt = synth.default_opt((7, 7), gnn_inc_glob_feat_f=True, gnn_normalize=True)
    with pytest.raises(NotImplementedError, match="global CNN features"):
        DeformerTrainer(cuda_model(synth.SyntheticDataset(2, (7, 7)), opt))
    opt = synth.default_opt((7, 7), gnn_dont_train=True, **TEMP)
    with pytest.raises(NotImplementedError, match="gnn_dont_train"):
        DeformerTrainer(cuda_model(synth.SyntheticDataset(2, (7, 7)), opt))
    opt = synth.default_opt((60, 60), **TEMP)
    tr = DeformerTrainer(cuda_model(synth.SyntheticDataset(2, (60, 60)), opt), use_cuda_graph=False)
    with pytest.raises(NotImplementedError, match="mesh-resident"):
        tr.add_batch(synth.make_batch((60, 60), 2, seed=1))
    assert not tr.slots
    opt = synth.default_opt((7, 7), **TEMP)
    tr = DeformerTrainer(cuda_model(synth.SyntheticDataset(2, (7, 7)), opt, gad_force_stream=True), use_cuda_graph=False)
    with pytest.raises(NotImplementedError, match="mesh-resident"):
        tr.add_batch(synth.make_batch((7, 7), 2, seed=1))
    # gnn_normalize keeps every route, the streaming launch chain and the cluster kernel included
    for md, extra in (((7, 7), dict(gad_force_stream=True)), ((60, 60), {})):
        opt, ds, data, state = _case(md, 2, **NORM)
        model, tr = _trainer(ds, opt, state, **extra)
        sid = tr.add_batch(data)
        loss = _step_without_optimizer(tr, sid)
        x_phys, want = _module_loss(opt, cuda_model(ds, opt, state, gad_store_alpha=False, **extra), data)
        assert util.rel_err(tr.slots[sid].x_phys, x_phys.reshape(-1, 2)) <= 1e-5
        assert abs(loss - want.item()) <= 1e-5 * want.item()


def test_c_abi_rejects_bad_arguments():
    lib = _lib.load()
    buf = torch.zeros(4096, device="cuda")
    p = buf.data_ptr()
    for args in ((None, 8, p), (p, 8, None), (p, 0, p), (p, -3, p)):
        assert lib.gad_batch_max(*args, None) == 1
        assert "gad_batch_max" in lib.gad_last_error().decode()
    for args, word in (((None, p, 1, 4, p), "null"), ((p, None, 1, 4, p), "null"), ((p, p, 1, 4, None), "null"),
                       ((p, p, 0, 4, p), "Lw=0"), ((p, p, 1, 3, p), "CE=3")):
        assert lib.gad_temp_fold(*args, None) == 1
        assert word in lib.gad_last_error().decode()
    for args, word in (((None, p, p, 1, 4, p, p), "null"), ((p, p, None, 1, 4, p, p), "null"),
                       ((p, p, p, 1, 4, None, p), "null"), ((p, p, p, 1, 4, p, None), "null"),
                       ((p, p, p, -1, 4, p, p), "Lw=-1"), ((p, p, p, 2, 16, p, p), "CE=16")):
        assert lib.gad_temp_fold_bwd(*args, None) == 1
        assert word in lib.gad_last_error().decode()
    torch.cuda.synchronize()


def test_kernels_match_torch():
    """gad_batch_max is torch.max (sign, -0 / +0 and NaN included); gad_temp_fold and gMu_base equal the module's torch
    expressions bit for bit; g_temp is within 1e-6 of them (torch sums in its own order)."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(0)
    out = torch.zeros(1, device="cuda")
    cases = [torch.randn(230400, generator=g), -torch.rand(5000, generator=g) - 1.0, torch.tensor([-0.0, -3.0]),
             torch.tensor([-0.0, 0.0, -1.0]), torch.randn(1000, generator=g) * 1e30, torch.tensor([7.0])]
    nan = torch.randn(70000, generator=g)
    nan[12345] = float("nan")
    for x in cases + [nan, -nan.abs()]:
        x = x.cuda()
        _lib.check(lib.gad_batch_max(x.data_ptr(), x.numel(), out.data_ptr(), None), "gad_batch_max")
        want = torch.max(x)
        assert (torch.isnan(want) and torch.isnan(out[0])) or out[0].item() == want.item(), (out, want)
    for Lw, CE in ((1, 4), (3, 4), (2, 2), (16, 8)):
        S = CE * CE + CE
        Mu = torch.randn(Lw, S, generator=g).cuda()
        temp = (torch.rand(Lw, generator=g) * 3 + 0.1).cuda()
        gMu = torch.randn(Lw, S, generator=g).cuda()
        Mu_eff, gMu_base, g_temp = torch.empty_like(Mu), torch.empty_like(Mu), torch.empty(Lw, device="cuda")
        _lib.check(lib.gad_temp_fold(Mu.data_ptr(), temp.data_ptr(), Lw, CE, Mu_eff.data_ptr(), None), "gad_temp_fold")
        _lib.check(lib.gad_temp_fold_bwd(gMu.data_ptr(), Mu_eff.data_ptr(), temp.data_ptr(), Lw, CE, gMu_base.data_ptr(),
                                         g_temp.data_ptr(), None), "gad_temp_fold_bwd")
        want_eff = Mu * (1.0 / temp.float().reshape(-1, 1))           # functional.DeformFunction.forward
        assert torch.equal(Mu_eff, want_eff)
        assert torch.equal(gMu_base, gMu / temp.reshape(-1, 1))       # DeformFunction.backward
        want_t = -(gMu * want_eff).sum(dim=1) / temp
        assert (g_temp - want_t).abs().max().item() <= 1e-6 * want_t.abs().max().item()


# 7 ------------------------------------------------------------------------------------------------------------------
def test_loopback_routes():
    """Single-process self-test of the data-parallel routes: a normalised slot keeps the in-kernel peer route and skips the
    collective of its maxima; a learnable-temperature slot takes the NCCL route."""
    md = (7, 7)
    for over, peer in ((NORM, True), (BOTH, False)):
        opt, ds, data, state = _case(md, 3, **over)
        model, tr = _trainer(ds, opt, state, gad_peer_loopback=(2, 1))
        sid = tr.add_batch(data)
        s = tr.slots[sid]
        assert s.norm and s.peer_route == peer and tr._one_launch(s) == peer and s.count_global == 2 * 3 * 49 * 2
        _step_without_optimizer(tr, sid)          # no process group: the maxima stay local
        assert s.f_scale.item() == data.f_tensor.max().item()
        tr.close()


@pytest.mark.timeout(300)
def test_two_gpus_match_one_gpu_on_the_union_batch(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, B, steps = 2, 3, 6
    out = tmp_path / "dp_norm_temp.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29541",
           os.path.join(ROOT, "tests", "dp_norm_temp_worker.py"), str(out), str(steps), str(B)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads(out.read_text())
    md = (12, 12)
    for key, over in (("normalize", NORM), ("normalize_learnable_a", BOTH)):
        got = res[key]
        assert got["ranks_equal"] and got["selfcheck"]["ranks_equal"] and got["shard_max_differ"]
        opt = synth.default_opt(md, lr=1e-2, **over)
        torch.manual_seed(42)
        model = cuda_model(synth.SyntheticDataset(2, md), opt, gad_store_alpha=False)
        tr = DeformerTrainer(model, lr=1e-2)
        sids = [tr.add_batch(_scale_features(synth.make_batch(md, world * B, seed=7, first_mesh_id=k * world * B),
                                             world * B, k * world * B)) for k in range(2)]
        for k in range(steps):
            tr.step(sids[k % 2])
        tr.synchronize()
        want = tr.flat.cpu()
        flat = torch.tensor(got["flat"])
        live = torch.ones(want.numel(), dtype=torch.bool)
        o = (tr.bk.data_ptr() - tr.flat.data_ptr()) // 4
        live[o:o + tr.bk.numel()] = False            # lin_key.bias: analytically zero gradient
        err = (flat - want)[live].abs().max().item() / want[live].abs().max().item()
        assert err <= 2e-3, (key, err)
