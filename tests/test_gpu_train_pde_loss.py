"""DeformerTrainer with loss_type='pde_loss' -- the reference's Poisson preset (params.py:109; src/run_GNN.py:109-110):
loss = mse(FEM solution on the deformed meshes, u_true_fine).

A step on a pde slot is a chain of library kernels: deformer forward (gad_deform_fwd_ell_raw) -> FEM forward
(gad_fem1d_fwd / gad_fem2d_fwd) -> gad_pde_loss -> FEM backward -> deformer backward -> weight gradients -> Adam.  These
are the kernels GNN.forward + autograd run for the same batch, so on identical parameters the trainer reproduces the
module path bit for bit: x_phys, the solution, the FEM cotangent handed to the deformer and the parameter gradients.
That is the check that matters here: the FEM gradient is a discontinuous function of the mesh points (DESIGN
section 11), so parity has to be shown on identical inputs, not against a path that rounds differently.

One link is not bit-reproducible by construction: the 2-D FEM backward (csrc/fem2d.cu) accumulates the gradient with
respect to the mesh points in fp64 shared-memory atomics, whose order is not fixed, so two runs of it on the same input
may differ in the last bit of the fp32 result.  The 2-D cotangent is therefore compared within 1e-6 of its largest
entry, and the parameter gradient as the deformer backward of the trainer's own cotangent (bit for bit).  The 1-D FEM
has no atomics and is compared bit for bit throughout."""
import copy
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gad_testutil as util
from g_adaptivity_b200 import _lib, synth
from g_adaptivity_b200.trainer import DeformerTrainer
from oracle import fem1d_oracle as F1
from oracle import gnn_oracle
from test_gpu_parity import cuda_model
from test_pde2d_golden import GOLDEN as GOLDEN_PDE2D, _rebuild

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _case(md, B, Q=101, K=101, seed=5, **over):
    """opt, dataset, batch and initial parameters of a pde_loss case (2-D: Q x Q fine mesh; 1-D: Q points)."""
    two_d = len(md) == 2
    opt = synth.default_opt(md, eval_quad_points=Q, load_quad_points=K, loss_type="pde_loss", **over)
    ds = synth.SyntheticDataset(len(md), md, eval_quad_points=Q if two_d else None)
    if ds.x_comp_shared is None:
        ds.x_comp_shared = synth.make_batch(md, 1).x_comp
    data = synth.make_batch(md, B, seed=seed, eval_quad_points=Q, with_u_true_fine=two_d)
    torch.manual_seed(42)
    state = copy.deepcopy(gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict())
    return opt, ds, data, state


def _module_step(ds, opt, state, data, retain_graph=False):
    """GNN.forward + mse(sol, u_true_fine) + autograd: (model, x_phys with its gradient, sol, loss)."""
    m = cuda_model(ds, opt, state, gad_store_alpha=False)
    m.train()
    _, x_phys, sol = m(data)
    x_phys.retain_grad()
    loss = F.mse_loss(sol, data.u_true_fine_tensor.cuda())
    loss.backward(retain_graph=retain_graph)
    return m, x_phys, sol, loss


def _step_without_optimizer(tr, sid):
    with torch.cuda.stream(tr.stream):
        tr._issue(tr.slots[sid], tr.stream.cuda_stream, with_optimizer=False)
    tr.synchronize()
    return tr.slots[sid].loss.item()


def _module_grads(m):
    return {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}


def _check_links(ds, opt, state, data, s, trainer_model, same_tiles: bool = True):
    """The module path at parameters `state` against the trainer's last step on slot `s`, link by link on identical
    inputs: x_phys and the solution bit for bit; the FEM cotangent handed to the deformer bit for bit (1-D) or within
    1e-6 of its largest entry (2-D, see the module docstring); the module's deformer backward of the TRAINER's
    cotangent against the trainer's gradient (_compare_grads).  Returns the module's loss and how the gradients
    compared."""
    m, x_phys, sol, loss = _module_step(ds, opt, state, data, retain_graph=True)
    assert torch.equal(s.x_phys.reshape(-1), x_phys.detach().reshape(-1))
    assert torch.equal((s.sol if s.order is None else s.sol.index_select(1, s.order.long())).reshape(-1), sol.detach())
    cot, cot_m = s.g_out.reshape(-1), x_phys.grad.reshape(-1)
    if not torch.equal(cot, cot_m):
        assert opt["mesh_dims"] and len(opt["mesh_dims"]) == 2, "the 1-D FEM cotangent must be bit-identical"
        assert (cot - cot_m).abs().max().item() <= 1e-6 * cot_m.abs().max().item()
    m.zero_grad(set_to_none=True)
    x_phys.backward(s.g_out.reshape(x_phys.shape))
    return loss, _compare_grads(trainer_model, _module_grads(m), same_tiles)


def _compare_grads(trainer_model, want, same_tiles: bool):
    """The trainer's gradient (views of its flat gradient) against the module's .grad: bit for bit when both ran the
    deformer backward on the same tiles, otherwise within 1e-6 of the largest entry."""
    got = {n: p.grad for n, p in trainer_model.named_parameters() if n in want}
    assert sorted(got) == sorted(want)
    if same_tiles:
        for n in want:
            assert torch.equal(got[n], want[n]), n
        return "bit-identical (same tiles)"
    scale = max(g.abs().max().item() for g in want.values())
    worst = max((got[n] - want[n]).abs().max().item() for n in want) / scale
    assert worst <= 1e-6, worst
    return f"within {worst:.1e} of the largest entry (different tiles)"


# 1 ------------------------------------------------------------------------------------------------------------------
ROWS = [
    ((7, 7), 3, dict(Q=13, K=9)),
    ((7, 7), 3, dict(Q=13, K=9, ode_method="rk4")),
    ((7, 7), 3, dict(Q=13, K=9, share_conv=False, num_layers=3)),
    ((7, 7), 3, dict(Q=13, K=9, learn_step=True)),
    ((30, 30), 16, dict()),
    ((30, 30), 16, dict(ode_method="rk4", share_conv=False)),
    ((30, 30), 256, dict()),
    ((200,), 64, dict()),
    ((200,), 64, dict(ode_method="rk4")),
    ((200,), 64, dict(learn_step=True, share_conv=False)),
]


def _row_id(r):
    md, B, over = r
    extra = "-".join(f"{k}={v}" for k, v in over.items() if k not in ("Q", "K"))
    return "x".join(map(str, md)) + f"-B{B}" + (f"-{extra}" if extra else "")


@pytest.mark.parametrize("row", ROWS, ids=[_row_id(r) for r in ROWS])
def test_one_step_matches_the_module_path_bit_for_bit(row):
    md, B, over = row
    opt, ds, data, state = _case(md, B, **over)
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert s.pde and not tr._one_launch(s)
    got_loss = _step_without_optimizer(tr, sid)
    same_tiles = torch.equal(s.graph.ell_tile_ptr, cuda_model(ds, opt)._graph(data, tr.dev, True).ell_tile_ptr)
    loss, how = _check_links(ds, opt, state, data, s, model, same_tiles)
    assert abs(got_loss - loss.item()) <= 1e-6 * abs(loss.item()), (got_loss, loss.item())
    print(_row_id(row), "gradient:", how)


# 2 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", GOLDEN_PDE2D, ids=[os.path.basename(p)[:-3] for p in GOLDEN_PDE2D])
def test_one_step_matches_the_reference_fixture_2d(path):
    """Bars of test_pde2d_golden.py::test_cuda_pde_loss_2d_matches_reference_fixture."""
    fx = torch.load(path)
    opt, ds, data, md, B, Q = _rebuild(fx)
    model = cuda_model(ds, opt, fx["state_dict"], gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    loss = _step_without_optimizer(tr, sid)
    sc = fx["coeffs"].abs().max().item()
    assert (s.x_phys.cpu() - fx["x_phys"]).abs().max().item() <= 1e-5 * fx["x_phys"].abs().max().item()
    sol = s.sol.index_select(1, s.order.long()).reshape(-1)
    assert (sol.cpu() - fx["sol"]).abs().max().item() <= 2e-5 * sc
    assert abs(loss - fx["loss"]) <= 1e-4 * abs(fx["loss"])
    scale = max(g.abs().max().item() for k, g in fx["grads"].items() if "lin_key.bias" not in k)
    worst = max((p.grad.cpu() - fx["grads"][k]).abs().max().item() / scale
                for k, p in model.named_parameters() if k in fx["grads"] and "lin_key.bias" not in k)
    assert worst <= 5e-2, worst


def test_one_step_matches_the_fp64_oracle_1d():
    """Bars of test_fem1d.py::test_pde_loss_through_the_deformer_1d (loss 1e-4, solution 1e-5, gradients 1e-3)."""
    md, B = (21,), 5
    opt, ds, data, state = _case(md, B, seed=3)
    ref = gnn_oracle.GNNRef(ds, copy.deepcopy(synth.default_opt(md))).double()
    ref.load_state_dict({k: v.double() for k, v in state.items()})
    d64 = data.clone()
    for k in d64.keys():
        v = getattr(d64, k)
        if torch.is_tensor(v) and v.dtype == torch.float32:
            setattr(d64, k, v.double())
    xp = ref(d64).squeeze(-1)
    Q, K, n = opt["eval_quad_points"], opt["load_quad_points"], md[0]
    quad = torch.linspace(0, 1, Q, dtype=torch.float32).double()
    sols = []
    for b in range(B):
        cs = [torch.tensor(float(np.asarray(c).reshape(-1)[0]), dtype=torch.float64) for c in data.pde_params["centers"][b]]
        ss = [torch.tensor(float(np.asarray(s).reshape(-1)[0]), dtype=torch.float64) for s in data.pde_params["scales"][b]]
        _, sol, *_ = F1.torch_fem_1d(xp[b * n:(b + 1) * n], quad, cs, ss, load_quad_points=K)
        sols.append(sol)
    sol_ref = torch.cat(sols)
    loss_ref = F.mse_loss(sol_ref, data.u_true_fine_tensor.double())
    loss_ref.backward()
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(data)
    loss = _step_without_optimizer(tr, sid)
    s = tr.slots[sid]
    assert abs(loss - loss_ref.item()) <= 1e-4 * abs(loss_ref.item())
    assert (s.sol.reshape(-1).cpu().double() - sol_ref.detach()).abs().max().item() <= 1e-5 * sol_ref.abs().max().item()
    scale = max(p.grad.abs().max().item() for n_, p in ref.named_parameters() if p.grad is not None and "lin_key.bias" not in n_)
    got = dict(model.named_parameters())
    for n_, q in ref.named_parameters():
        if q.grad is None or "lin_key.bias" in n_:
            continue
        err = (got[n_].grad.cpu().double() - q.grad).abs().max().item() / max(q.grad.abs().max().item(), 1e-3 * scale)
        assert err <= 1e-3, (n_, err)


# 3 ------------------------------------------------------------------------------------------------------------------
K_STEPS, LR = 10, 1e-3


def _module_adam(ds, opt, state, batches, lr=LR):
    m = cuda_model(ds, opt, state, gad_store_alpha=False)
    m.train()
    optim = torch.optim.Adam(m.parameters(), lr=lr)
    losses = []
    for k in range(K_STEPS):
        data = batches[k % len(batches)]
        optim.zero_grad(set_to_none=True)
        _, _, sol = m(data)
        loss = F.mse_loss(sol, data.u_true_fine_tensor.cuda())
        loss.backward()
        optim.step()
        losses.append(float(loss.item()))
    return {n: p.detach().cpu().clone() for n, p in m.named_parameters()}, losses


def _trainer_run(ds, opt, state, batches, mode, lr=LR, check_grads=False):
    """K steps in `mode` (eager / graph / epoch).  With check_grads (eager, graph): before every step the module path
    is run at the trainer's current parameters, and the step's gradient must equal it bit for bit."""
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, lr=lr, use_cuda_graph=(mode != "eager"))
    sids = [tr.add_batch(b) for b in batches]
    losses = []
    if mode == "epoch":
        for _ in range(K_STEPS // len(sids)):
            tr.run_epoch(sids)
            tr.synchronize()
            losses += [float(tr.slots[s].loss.item()) for s in sids]
    else:
        for k in range(K_STEPS):
            tr.synchronize()
            cur = {n: v.detach().clone() for n, v in model.state_dict().items()} if check_grads else None
            l = tr.step(sids[k % len(sids)])
            tr.synchronize()
            losses.append(float(l.item()))
            if check_grads:         # the step's gradient against the module path at the parameters it started from
                _check_links(ds, opt, cur, batches[k % len(sids)], tr.slots[sids[k % len(sids)]], model)
    assert int(tr.step_count.item()) == K_STEPS
    return tr, {n: p.detach().cpu().clone() for n, p in model.named_parameters()}, losses


def _compare_params(got, want, losses, ref_losses, tol=2e-3):
    """After K Adam steps: the project's Adam bar, 2e-3 of the largest parameter (lin_key.bias excluded: its gradient
    is analytically zero, so Adam turns rounding noise into O(lr)); torch.optim.Adam and gad_adam_step round apart."""
    names = [n for n in want if "lin_key.bias" not in n]
    scale = max(want[n].abs().max().item() for n in names)
    worst = max((got[n] - want[n]).abs().max().item() for n in names) / scale
    print(f"parameters after {K_STEPS} Adam steps: max |trainer - module| / max |param| = {worst:.3e}")
    assert worst <= tol, worst
    assert abs(losses[0] - ref_losses[0]) <= 1e-6 * abs(ref_losses[0])
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 2e-3 * abs(b), (losses, ref_losses)


@pytest.fixture(scope="module", params=["2d", "1d"])
def adam_case(request):
    if request.param == "2d":
        md, B, over = (7, 7), 4, dict(Q=13, K=9)
    else:
        md, B, over = (200,), 32, dict()
    opt, ds, _, state = _case(md, B, **over)
    Q = over.get("Q", 101)
    batches = [synth.make_batch(md, B, seed=31, first_mesh_id=r * B, eval_quad_points=Q, with_u_true_fine=len(md) == 2)
               for r in range(2)]
    want, ref_losses = _module_adam(ds, opt, state, batches)
    return opt, ds, batches, state, want, ref_losses


@pytest.mark.parametrize("mode", ["eager", "graph", "epoch"])
def test_k_adam_steps_match_the_module_path(adam_case, mode):
    opt, ds, batches, state, want, ref_losses = adam_case
    tr, got, losses = _trainer_run(ds, opt, state, batches, mode, check_grads=mode != "epoch")
    _compare_params(got, want, losses, ref_losses)
    if mode == "epoch":       # one graph for the whole pass: the same parameters as step by step, bit for bit
        _, got_eager, losses_eager = _trainer_run(ds, opt, state, batches, "eager")
        assert losses == losses_eager and all(torch.equal(got[n], got_eager[n]) for n in got)


# 4 ------------------------------------------------------------------------------------------------------------------
GLOB_ROWS = [
    ((12, 12), 5, dict(gnn_inc_glob_feat_f=True, gnn_inc_glob_feat_uu=True)),
    ((30, 30), 3, dict(gnn_inc_glob_feat_f=True, gnn_inc_glob_feat_uu=True, hidden_dim=16)),
    ((200,), 16, dict(gnn_inc_glob_feat_f=True, gnn_inc_glob_feat_uu=True)),
]


@pytest.mark.parametrize("row", GLOB_ROWS, ids=[_row_id(r) for r in GLOB_ROWS])
def test_global_cnn_features_one_step(row):
    """Bars of test_gpu_train_glob_features.py (coordinates and loss 1e-5, gradients 2e-4): the module computes the
    bias offset with torch ops, the trainer with gad_glob_bias_fwd, so they round apart."""
    md, B, over = row
    opt, ds, data, state = _case(md, B, **over)
    model = cuda_model(ds, opt, state, gad_store_alpha=False)
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert s.glob and s.pde and model.n_glob_used > 0
    got_loss = _step_without_optimizer(tr, sid)
    m, x_phys, _, loss = _module_step(ds, opt, state, data, retain_graph=True)
    assert util.rel_err(s.x_phys.reshape(-1), x_phys.reshape(-1)) <= 1e-5
    assert abs(got_loss - loss.item()) <= 1e-5 * abs(loss.item())
    # x_phys differs in the last bits (the bias offset is rounded apart), and the FEM gradient is discontinuous in the
    # mesh points: the deformer + CNN backward is compared on the trainer's own FEM cotangent
    m.zero_grad(set_to_none=True)
    x_phys.backward(s.g_out.reshape(x_phys.shape))
    want = _module_grads(m)
    got = {n: p.grad for n, p in model.named_parameters() if n in want}
    assert any("global_feature" in n for n in got)
    scale = max(g.abs().max().item() for n, g in want.items() if "lin_key.bias" not in n)
    for n, g in want.items():
        if "lin_key.bias" in n:
            continue
        err = (got[n].double() - g.double()).abs().max().item() / max(g.abs().max().item(), 1e-2 * scale)
        assert err <= 2e-4, (n, err)


@pytest.mark.parametrize("row", [GLOB_ROWS[0], GLOB_ROWS[2]], ids=[_row_id(GLOB_ROWS[0]), _row_id(GLOB_ROWS[2])])
def test_global_cnn_features_k_adam_steps(row):
    md, B, over = row
    opt, ds, _, state = _case(md, B, **over)
    batches = [synth.make_batch(md, B, seed=31, first_mesh_id=r * B, with_u_true_fine=len(md) == 2) for r in range(2)]
    want, ref_losses = _module_adam(ds, opt, state, batches)
    _, got, losses = _trainer_run(ds, opt, state, batches, "graph")
    assert any("global_feature" in n for n in got)
    _compare_params(got, want, losses, ref_losses)


# 5 ------------------------------------------------------------------------------------------------------------------
def test_steps_are_bit_reproducible_on_every_route():
    """On 1-D meshes: the 2-D FEM backward's fp64 shared-memory atomics leave the last bit of its result to the order
    of the adds (module docstring), which no route of the trainer can fix."""
    md, B = (200,), 16
    opt, ds, _, state = _case(md, B)
    batches = [synth.make_batch(md, B, seed=50 + k) for k in range(2)]
    for b in batches:
        b.pin_memory()
    runs = [_trainer_run(ds, opt, state, batches, "graph") for _ in range(2)]
    assert runs[0][2] == runs[1][2] and torch.equal(runs[0][0].flat, runs[1][0].flat)

    outs = []
    for mode in ("step", "train_batch", "packed_native", "packed_prefix_native", "python_loop"):
        model = cuda_model(ds, opt, state, gad_store_alpha=False)
        tr = DeformerTrainer(model, lr=LR)
        if mode == "train_batch":
            losses = []
            for k in range(6):
                l = tr.train_batch(batches[k % 2], ring=2)
                with torch.cuda.stream(tr.stream):            # the loss is written on the trainer's stream
                    losses.append(l.clone())
            tr.synchronize()
            losses = torch.stack([x.cpu() for x in losses]).reshape(-1)
            outs.append((mode, losses, tr.flat.clone().cpu()))
            continue
        sids = [tr.add_batch(b) for b in batches]
        if mode == "step":
            losses = []
            for k in range(6):
                l = tr.step(sids[k % 2])
                with torch.cuda.stream(tr.stream):
                    losses.append(l.clone())
            tr.synchronize()
            losses = torch.stack([x.cpu() for x in losses]).reshape(-1)
        elif mode in ("packed_native", "packed_prefix_native"):
            full = mode == "packed_native"
            src = [tr.pack_host(sid, b, with_x_comp=full) for sid, b in zip(sids, batches)]
            if not full:
                assert src[0].numel() == tr.slots[sids[0]].in_offs[-1]
            losses = tr.run_from_host(src, 6, native=True).clone()
        else:
            losses = tr.run_from_host(batches, 6, native=False).clone()
        outs.append((mode, losses, tr.flat.clone().cpu()))
    for mode, losses, flat in outs[1:]:
        assert torch.equal(outs[0][1], losses) and torch.equal(outs[0][2], flat), mode


# 6 ------------------------------------------------------------------------------------------------------------------
def test_refusals():
    opt, ds, data, _ = _case((7, 7), 2, Q=13, K=9)
    tr = DeformerTrainer(cuda_model(ds, opt, gad_store_alpha=False), use_cuda_graph=False)
    with pytest.raises(NotImplementedError, match="equal size"):
        tr.add_batch(synth.make_mixed_batch([(6, 6), (7, 7)], seed=1))
    with pytest.raises(NotImplementedError, match="mesh-resident"):
        DeformerTrainer(cuda_model(ds, opt, gad_store_alpha=False, gad_force_stream=True),
                        use_cuda_graph=False).add_batch(data)
    for attr in ("mesh", "mapping_tensor_fine"):
        ds2 = synth.SyntheticDataset(2, (7, 7), eval_quad_points=13)
        setattr(ds2, attr, None)
        with pytest.raises(ValueError, match=attr):
            DeformerTrainer(cuda_model(ds2, opt, gad_store_alpha=False), use_cuda_graph=False).add_batch(data)
    # what the FEM kernels reject is refused by add_batch, before any capture
    opt17, ds17, _, _ = _case((7, 7), 2, Q=13, K=9)
    many = synth.make_batch((7, 7), 2, seed=1, num_gauss=17, eval_quad_points=13, with_u_true_fine=True)
    with pytest.raises(RuntimeError, match="Gaussians"):
        DeformerTrainer(cuda_model(ds17, opt17, gad_store_alpha=False), use_cuda_graph=False).add_batch(many)
    opt39, ds39, big, _ = _case((39, 39), 1, Q=13, K=9)
    tr39 = DeformerTrainer(cuda_model(ds39, opt39, gad_store_alpha=False), use_cuda_graph=False)
    with pytest.raises((RuntimeError, NotImplementedError), match="fem2d|mesh-resident"):
        tr39.add_batch(big)
    assert not tr39.slots and not tr39.graphs
    with pytest.raises(NotImplementedError):
        DeformerTrainer(cuda_model(ds, dict(opt, ode_method="rk4", learn_step=True)))
    with pytest.raises(NotImplementedError):
        cuda_model(ds, dict(opt, data_type="randg_mix"))


def test_explicit_loss_fn_still_trains_the_mesh_loss():
    opt, ds, data, state = _case((7, 7), 3, Q=13, K=9)
    tr = DeformerTrainer(cuda_model(ds, opt, state, gad_store_alpha=False), loss_fn="l1", use_cuda_graph=False)
    sid = tr.add_batch(data)
    assert not tr.pde and not tr.slots[sid].pde and tr._one_launch(tr.slots[sid])
    mesh = dict(opt, loss_type="mesh_loss")
    tr2 = DeformerTrainer(cuda_model(ds, mesh, state, gad_store_alpha=False), use_cuda_graph=False)
    sid2 = tr2.add_batch(data)
    for t, i in ((tr, sid), (tr2, sid2)):
        t.step(i)
    tr.synchronize(), tr2.synchronize()
    assert torch.equal(tr.slots[sid].loss, tr2.slots[sid2].loss) and torch.equal(tr.flat, tr2.flat)


def test_c_abi_rejects_bad_arguments():
    lib = _lib.load()
    buf = torch.zeros(4096, device="cuda")
    p = buf.data_ptr()
    ws = lib.gad_pde_loss_workspace_bytes(2, 8)
    assert 0 < ws <= buf.numel() * 4
    for args, word in [((None, None, p, 2, 8, 1.0, p, p, p), "NULL"), ((p, None, None, 2, 8, 1.0, p, p, p), "NULL"),
                       ((p, None, p, 2, 8, 1.0, None, p, p), "NULL"), ((p, None, p, 2, 8, 1.0, p, p, None), "NULL"),
                       ((p, None, p, 0, 8, 1.0, p, p, p), "positive"), ((p, None, p, 2, -1, 1.0, p, p, p), "positive"),
                       ((p, None, p, 2, 8, float("nan"), p, p, p), "finite")]:
        assert lib.gad_pde_loss(*args, None) == 1          # GAD_ERR_ARG
        assert word in lib.gad_last_error().decode()
    assert lib.gad_pde_loss(p, None, p, 2, 8, 0.125, p, None, p + 8192, None) == 0      # g_sol may be NULL
    torch.cuda.synchronize()


def test_loss_kernel_matches_torch_mse_bit_for_bit():
    """gad_pde_loss on its own: the cotangent is torch's mse_loss backward bit for bit, through the index map too."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(0)
    B, Q = 37, 169
    sol = torch.randn(B, Q, generator=g).cuda()
    tgt = torch.randn(B * Q, generator=g).cuda()
    order = torch.randperm(Q, generator=g).cuda()
    for idx in (None, order):
        ref_in = (sol if idx is None else sol.index_select(1, idx)).reshape(-1).clone().requires_grad_(True)
        ref = F.mse_loss(ref_in, tgt)
        ref.backward()
        want = torch.zeros_like(sol)
        want[:, idx if idx is not None else torch.arange(Q, device="cuda")] = ref_in.grad.view(B, Q)
        loss, g_sol = torch.zeros(1, device="cuda"), torch.full_like(sol, float("nan"))
        ws = torch.empty(lib.gad_pde_loss_workspace_bytes(B, Q), dtype=torch.uint8, device="cuda")
        o32 = None if idx is None else idx.to(torch.int32)
        _lib.check(lib.gad_pde_loss(sol.data_ptr(), _lib.ptr(o32), tgt.data_ptr(), B, Q, float(2.0 / (B * Q)),
                                    loss.data_ptr(), g_sol.data_ptr(), ws.data_ptr(), None), "gad_pde_loss")
        torch.cuda.synchronize()
        assert torch.equal(g_sol, want)
        assert abs(loss.item() - ref.item()) <= 1e-6 * ref.item()


# 7 ------------------------------------------------------------------------------------------------------------------
def test_loopback_slot_takes_the_nccl_route():
    opt, ds, data, _ = _case((7, 7), 3, Q=13, K=9)
    model = cuda_model(ds, opt, gad_store_alpha=False, gad_peer_loopback=(2, 1))
    tr = DeformerTrainer(model, use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert s.pde and not s.peer_route and not tr._one_launch(s) and s.count_global == 2 * 3 * 13 * 13


@pytest.mark.timeout(300)
def test_two_gpus_match_one_gpu_on_the_union_batch(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, B, steps = 2, 3, 6
    out = tmp_path / "dp_pde.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29539", os.path.join(ROOT, "tests", "dp_pde_worker.py"),
           str(out), str(steps), str(B)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads(out.read_text())
    assert res["ranks_equal"] and not res["peer_route"] and res["selfcheck"]["ranks_equal"]
    md, Q = (7, 7), 13
    opt = synth.default_opt(md, eval_quad_points=Q, load_quad_points=9, loss_type="pde_loss", lr=1e-2)
    ds = synth.SyntheticDataset(2, md, eval_quad_points=Q)
    torch.manual_seed(42)
    model = cuda_model(ds, opt, gad_store_alpha=False)
    tr = DeformerTrainer(model, lr=1e-2)
    sids = [tr.add_batch(synth.make_batch(md, world * B, seed=7, first_mesh_id=k * world * B, eval_quad_points=Q,
                                          with_u_true_fine=True)) for k in range(2)]
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
