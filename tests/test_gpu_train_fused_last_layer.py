"""The one-launch Euler training step (csrc/ell_kernels.cuh: k_ell_train<..., GAD_METHOD_EULER>) computes phase A
(the destination pass) of the last layer's backward inside the last forward layer, from the rows that layer gathered
(ell_math.cuh: ell_feval_bwd_dst), and starts tile_backward at phase B of that layer.

Against the unfused pass: the module kernels k_ell_fwd + k_ell_bwd on the same slot, fed the cotangent the train
kernel forms, give the same x_phys and the same per-tile gradient partials, bit for bit.  Against the launch chain
(gad_no_fused_train) within the bars of test_gpu_ell, against autograd through the oracle in fp64 within those of
test_gpu_train_rk4, and bit-identical under graph replay.
"""
import copy

import pytest
import torch

from g_adaptivity_b200 import _lib, dp, synth
from g_adaptivity_b200 import functional as GF
from g_adaptivity_b200.trainer import DeformerTrainer
from test_gpu_parity import cuda_model, grads_of, oracle_model
from test_gpu_train_rk4 import _oracle_loss_and_grads, _step_without_optimizer

import gad_testutil as util

pytestmark = pytest.mark.gpu


def _case(mesh_dims, B, seed=0, burgers=False, **over):
    opt = synth.burgers_opt(mesh_dims, **over) if burgers else synth.default_opt(mesh_dims, **over)
    ds = synth.SyntheticDataset(len(mesh_dims), mesh_dims)
    data = synth.make_batch(mesh_dims, B, seed=seed, burgers=burgers)
    torch.manual_seed(42)
    state = copy.deepcopy(oracle_model(ds, opt).state_dict())
    return opt, ds, data, state


def _unfused_partials(tr, s, loss_fn):
    """x_phys and the per-tile partials [G_M, G_u, g_tau] of the module kernels on slot `s`: k_ell_fwd, then k_ell_bwd
    (whose phase A is the separate destination pass) on the cotangent the train kernel forms from x_phys."""
    lib, P, g = _lib.load(), _lib.ptr, s.graph
    N, CE, L, Lw, dim = s.N, tr.CE, tr.L, tr.Lw, tr.dim
    dev = s.x_phys.device
    states = torch.empty((L, N, CE), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(lib.gad_pack_features(P(s.x_comp), P(s.f), P(s.uu), None, None, N, dim, CE, P(states), stream),
               "gad_pack_features")
    x_phys = GF.deform_forward(g, states[0], dim, tr.Mu, tr.tau, states=states)
    d = x_phys - s.target
    gs = dp.local_grad_scale(N * dim, s.count_global)
    g_x = torch.sign(d) * gs if loss_fn == "l1" else d * (2.0 * gs)   # the kernel's 2 * grad_scale * d (2x is exact)
    ws_bytes = lib.gad_ell_workspace_bytes(CE, g.T, L)
    ws = torch.zeros(ws_bytes // 4, dtype=torch.float32, device=dev)
    gMu = torch.empty_like(tr.Mu)
    g_tau = torch.empty(L, dtype=torch.float32, device=dev) if tr.gtau is not None else None
    _lib.check(lib.gad_deform_bwd_ell(P(g.ell_in), P(g.ell_out), N, P(g.ell_tile_ptr), g.T, g.max_tile_nodes, g.ell_deg,
                                      P(states), P(g_x), dim, CE, P(tr.Mu), None, Lw, P(tr.tau), L, P(gMu), P(g_tau),
                                      None, P(ws), ws_bytes, stream), "gad_deform_bwd_ell")
    torch.cuda.synchronize(dev)
    return x_phys, ws


def _check_bit_identical_to_the_unfused_pass(mesh_dims, B, burgers, over, loss_fn):
    opt, ds, data, state = _case(mesh_dims, B, seed=3, burgers=burgers, **over)
    model = cuda_model(ds, opt, state)
    tr = DeformerTrainer(model, loss_fn=loss_fn, use_cuda_graph=False)
    sid = tr.add_batch(data)
    s = tr.slots[sid]
    assert tr._fused_ell(s)
    _step_without_optimizer(tr, sid)
    T, L, CE = s.graph.T, tr.L, tr.CE
    nacc = CE * CE + CE + 1
    n_part = T * (L if tr.Lw > 1 else 1) * nacc
    got = s.bwd_ws.view(torch.float32)
    x_phys, ws = _unfused_partials(tr, s, loss_fn)
    assert torch.equal(s.x_phys, x_phys)
    assert torch.equal(got[:n_part], ws[:n_part])
    if tr.gtau is not None and tr.Lw == 1:       # g_tau partials [T, L]
        o = T * L * nacc
        assert torch.equal(got[o:o + T * L], ws[o:o + T * L])


@pytest.mark.parametrize("loss_fn", ["l1", "mse"])
@pytest.mark.parametrize("mesh_dims,B,burgers", [
    ((30, 30), 256, False),      # the benchmarked shape: ELL rows in shared memory
    ((50, 50), 1024, False),     # cfg-5 shape: ELL rows streamed from L2
    ((200,), 64, True),          # 1-D Burgers: CE = 2, a staged target of one float per node
])
def test_bit_identical_to_the_unfused_pass_at_production_shapes(mesh_dims, B, burgers, loss_fn):
    _check_bit_identical_to_the_unfused_pass(mesh_dims, B, burgers, {}, loss_fn)


@pytest.mark.parametrize("loss_fn", ["l1", "mse"])
@pytest.mark.parametrize("mesh_dims,B,burgers,over", [
    ((30, 30), 24, False, {"share_conv": False}),
    ((30, 30), 24, False, {"learn_step": True}),
    ((30, 30), 24, False, {"share_conv": False, "learn_step": True, "num_layers": 3}),
    ((30, 30), 24, False, {"num_layers": 1}),          # the fused layer is the only one: no source pass follows it
    ((30, 30), 24, False, {"num_layers": 2}),
    ((200,), 64, True, {"num_layers": 1}),
    ((200,), 64, True, {"learn_step": True, "num_layers": 2}),
])
def test_bit_identical_to_the_unfused_pass_with_options(mesh_dims, B, burgers, over, loss_fn):
    _check_bit_identical_to_the_unfused_pass(mesh_dims, B, burgers, over, loss_fn)


@pytest.mark.parametrize("over", [{}, {"num_layers": 1}, {"share_conv": False, "learn_step": True}])
def test_one_launch_equals_the_launch_chain(over):
    """The chain runs the CSR tile kernels (another softmax normalisation): bars of test_gpu_ell."""
    opt, ds, data, state = _case((30, 30), 24, seed=6, **over)
    res = []
    for no_fused in (False, True):
        model = cuda_model(ds, opt, state, gad_no_fused_train=no_fused)
        tr = DeformerTrainer(model, use_cuda_graph=False)
        sid = tr.add_batch(data)
        assert tr._fused_ell(tr.slots[sid]) != no_fused
        loss = _step_without_optimizer(tr, sid)
        res.append((loss, tr.gflat.clone().cpu(), tr.slots[sid].x_phys.clone().cpu()))
    assert abs(res[0][0] - res[1][0]) <= 1e-6 * abs(res[1][0])
    assert (res[0][1] - res[1][1]).abs().max().item() <= 1e-5 * res[1][1].abs().max().item()
    assert util.rel_err(res[0][2], res[1][2]) <= 2e-6


@pytest.mark.parametrize("loss_fn", ["l1", "mse"])
def test_one_launch_matches_autograd_through_the_oracle(loss_fn):
    opt, ds, data, state = _case((20, 20), 7, seed=3, num_layers=3, learn_step=True)
    model = cuda_model(ds, opt, state)
    tr = DeformerTrainer(model, loss_fn=loss_fn, use_cuda_graph=False)
    sid = tr.add_batch(data)
    assert tr._one_launch(tr.slots[sid])
    loss = _step_without_optimizer(tr, sid)
    l64, loss_tol, g64, floor, scale = _oracle_loss_and_grads(ds, opt, data, state, loss_fn)
    assert abs(loss - l64) <= loss_tol * abs(l64), (loss, l64, loss_tol)
    util.check_grads_conditioned(grads_of(model), g64, floor, scale, tol=1e-4)


def test_graph_replay_is_deterministic():
    opt, ds, data, state = _case((30, 30), 64, seed=8)
    finals = []
    for _ in range(2):
        model = cuda_model(ds, opt, state)
        tr = DeformerTrainer(model, lr=1e-2)
        sid = tr.add_batch(data)
        losses = []
        for _ in range(10):
            loss = tr.step(sid)
            with torch.cuda.stream(tr.stream):
                losses.append(loss.clone())
        tr.synchronize()
        finals.append(([float(x.item()) for x in losses], tr.flat.clone().cpu()))
    assert finals[0][0][-1] < finals[0][0][0]
    assert finals[0][0] == finals[1][0]
    assert torch.equal(finals[0][1], finals[1][1])
