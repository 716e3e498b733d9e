"""Global CNN features (gnn_inc_glob_feat_f / _uu) on meshes beyond one CTA: the per-mesh bias offset `du` on the
cluster-resident kernels (csrc/cl_kernels.cu) and the streaming ELL kernels (csrc/stream_ell.cu), and the CNN backward
with its gradient planes in the global workspace (csrc/glob_cnn.cu).

Against the oracle in fp64 at the bars of test_glob_features.py (coordinates 1e-5, every gradient 2e-4, widened to 4x
the fp32 oracle's own deviation where that is larger, as gad_testutil.check_grads_conditioned does), route by route; routes against each other; the persistent streaming forward against the launch chain bit for bit; determinism;
and the refusals that stay (the CSR kernels take no offset)."""
from __future__ import annotations

import copy

import pytest
import torch
import torch.nn.functional as F

import gad_testutil as util
from g_adaptivity_b200 import synth
from g_adaptivity_b200 import functional as GF
from oracle import cnn_oracle, gnn_oracle

pytestmark = pytest.mark.gpu

FU = {"gnn_inc_glob_feat_f": True, "gnn_inc_glob_feat_uu": True}


def _dataset(md):
    ds = synth.SyntheticDataset(len(md), md)
    if ds.x_comp_shared is None:
        ds.x_comp_shared = synth.make_batch(md, 1).x_comp
    return ds


def _to64(data):
    d64 = data.clone()
    for k in d64.keys():
        v = getattr(d64, k)
        if torch.is_tensor(v) and v.dtype == torch.float32:
            setattr(d64, k, v.double())
    return d64


def _run_module(md, B, over, extra=None, seed=9):
    """(model, x_phys, parameter gradients) of one forward + L1 backward of the CUDA module."""
    from test_gpu_parity import cuda_model
    opt = synth.default_opt(md, **over)
    ds = _dataset(md)
    data = synth.make_batch(md, B, seed=seed)
    torch.manual_seed(42)
    ref32 = gnn_oracle.GNNRef(ds, copy.deepcopy(opt))
    model = cuda_model(ds, opt, ref32.state_dict(), **(extra or {}))
    model.train()
    out = model(data)
    F.l1_loss(out, data.x_phys.cuda().reshape(out.shape)).backward()
    grads = {n: p.grad.detach().cpu().clone() for n, p in model.named_parameters() if p.grad is not None}
    return model, out.detach().cpu(), grads, (opt, ds, data, ref32)


def _oracle(opt, ds, data, ref32):
    """x_phys of the oracle in fp64, its parameter gradients in fp64, and per parameter the deviation of the fp32 oracle
    from them (gad_testutil.fp64_grads_and_noise_floor)."""
    ref = gnn_oracle.GNNRef(ds, copy.deepcopy(opt))
    ref.load_state_dict(ref32.state_dict())
    ref = ref.double()
    ref_out = ref(_to64(data)).detach()
    r32 = gnn_oracle.GNNRef(ds, copy.deepcopy(opt))
    r32.load_state_dict(ref32.state_dict())
    gnn_oracle.mesh_loss(r32(data), data.x_phys).backward()
    g32 = {n: p.grad for n, p in r32.named_parameters() if p.grad is not None}
    g64, floor, scale = util.fp64_grads_and_noise_floor(ds, opt, data, r32, g32)
    return ref_out, g64, floor, scale


def _check_grads(got, g64, floor, scale, tol=2e-4):
    """test_glob_features.py's bar (2e-4 of each gradient's size, at least 1e-3 of the largest) or, where summing over
    thousands of nodes in fp32 leaves the fp32 oracle itself further from the fp64 gradient, 4 x that deviation
    (gad_testutil.check_grads_conditioned: the kernels' ex2 / lg2 / rcp carry 4 ulp)."""
    assert all(n in got for n in g64 if "lin_key.bias" not in n and "lin_skip" not in n)
    util.check_grads_conditioned(got, {n: g for n, g in g64.items() if "lin_skip" not in n}, floor, scale, tol=tol)


@pytest.fixture
def env(monkeypatch):
    def set_env(d):
        for k, v in d.items():
            monkeypatch.setenv(k, v)
    return set_env


CASES = [
    # id, mesh dims, meshes, model options, module extras, environment, expected route
    ("cluster", (64, 64), 2, FU, {}, {"GAD_FWD_POLICY": "cluster"}, "cluster"),
    ("stream", (64, 64), 2, FU, {"gad_no_cluster": True}, {"GAD_FWD_POLICY": "stream"}, "stream"),
    ("stream_chain", (64, 64), 2, FU, {"gad_no_cluster": True}, {"GAD_FWD_POLICY": "stream", "GAD_WIDE_PERSIST": "0"},
     "stream"),
    ("force_stream", (12, 12), 3, FU, {"gad_force_stream": True}, {}, "tiles"),
    ("rk4_50", (50, 50), 2, dict(FU, ode_method="rk4", num_layers=2), {}, {}, "tiles"),
    ("rk4_64", (64, 64), 2, dict(FU, ode_method="rk4", num_layers=2), {}, {}, "cluster_or_stream"),
    ("unshared", (64, 64), 2, dict(FU, share_conv=False, num_layers=3), {}, {}, "cluster_or_stream"),
    ("hidden16", (64, 64), 2, dict(FU, hidden_dim=16), {}, {}, "cluster_or_stream"),
    ("learnable_a", (64, 64), 2, dict(FU, softmax_temp_type="learnable_a"), {}, {}, "cluster_or_stream"),
    ("1d", (4000,), 3, FU, {}, {}, "cluster_or_stream"),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_module_matches_oracle_beyond_one_cta(case, env):
    name, md, B, over, extra, envd, route = case
    env(envd)
    model, out, grads, ctx = _run_module(md, B, over, extra)
    assert model.n_glob_used > 0
    g = model.last_graph
    if route == "tiles":
        assert g.tile_ptr is not None and g.T == B
    else:
        assert g.tile_ptr is None
    if route == "cluster":
        assert g.cl_in is not None and getattr(g, "clf_in", None) is not None
    ref_out, g64, floor, scale = _oracle(*ctx)
    assert util.rel_err(out, ref_out) <= 1e-5
    assert any("global_feature" in n for n in g64)
    _check_grads(grads, g64, floor, scale)
    with torch.no_grad():                                        # inference path (no autograd node)
        assert util.rel_err(model(ctx[2]).cpu(), ref_out) <= 1e-5


def test_routes_agree(env):
    """One batch per pair of routes that can both run it: mesh-resident vs streaming (30x30), cluster vs streaming
    (64x64).  Coordinates 1e-5 of their size, gradients 2e-5 of the largest (test_gpu_parity.py's cross-route bar)."""
    pairs = [
        ((30, 30), 3, [({}, {}), ({"gad_force_stream": True}, {})]),
        ((64, 64), 2, [({}, {"GAD_FWD_POLICY": "cluster"}), ({"gad_no_cluster": True}, {"GAD_FWD_POLICY": "stream"})]),
    ]
    for md, B, routes in pairs:
        res = []
        for extra, envd in routes:
            env(envd)
            _, out, grads, _ = _run_module(md, B, FU, extra)
            res.append((out, grads))
        (o0, g0), (o1, g1) = res
        assert util.rel_err(o1, o0) <= 1e-5, md
        scale = max(float(g.abs().max()) for g in g0.values())
        for k in g0:
            assert float((g0[k] - g1[k]).abs().max()) <= 2e-5 * scale, (md, k)


def test_persistent_forward_equals_the_launch_chain_with_du(env):
    """k_wide_persist against the chain of k_wide_stage launches, Euler and RK4, with the bias offset: same bits."""
    md, B = (64, 64), 2
    for method in ("euler", "rk4"):
        outs = []
        for persist in ("1", "0"):
            env({"GAD_FWD_POLICY": "stream", "GAD_WIDE_PERSIST": persist})
            from test_gpu_parity import cuda_model
            opt = synth.default_opt(md, ode_method=method, **FU)
            torch.manual_seed(42)
            model = cuda_model(_dataset(md), opt, None, gad_no_cluster=True)
            data = synth.make_batch(md, B, seed=3)
            with torch.no_grad():
                outs.append(model(data).cpu())
            g = model.last_graph
            assert g.tile_ptr is None
            if persist == "1":
                assert g.N <= g.persist_nodes(model.CE)
        assert torch.equal(outs[0], outs[1]), method


def test_streaming_kernels_take_du_null_as_before():
    """du = 0 gives the bits of du = None on the cluster and streaming routes (the offset is added to u before the
    products, and 0 changes nothing)."""
    from test_gpu_parity import cuda_model
    md, B = (64, 64), 2
    opt = synth.default_opt(md)
    torch.manual_seed(42)
    model = cuda_model(_dataset(md), opt)
    data = synth.make_batch(md, B, seed=4)
    with torch.no_grad():
        model(data)
    g = model.last_graph
    CE, dim = model.CE, model.dim
    dev = torch.device("cuda")
    Mu = model._folded_weights(dev)
    tau = model._tau(dev).float().contiguous()
    du0 = torch.zeros((B, Mu.shape[0], CE), device=dev)
    x_comp, f, uu = data.x_comp.cuda(), data.f_tensor.cuda(), data.uu_tensor.cuda()
    for method in (GF.METHOD_EULER, GF.METHOD_RK4):
        a = GF.deform_forward_raw(g, x_comp, f, uu, None, None, dim, CE, Mu, tau, method)
        b = GF.deform_forward_raw(g, x_comp, f, uu, None, None, dim, CE, Mu, tau, method, du=du0)
        assert torch.equal(a, b)
    L = int(tau.numel())
    states = torch.empty((L, g.N, CE), device=dev)
    GF.deform_forward_raw(g, x_comp, f, uu, None, None, dim, CE, Mu, tau, GF.METHOD_EULER, states=states)
    gx = torch.randn(g.N, dim, device=dev)
    for force in (False, True):       # cluster, then streaming (tile-less graph: force_stream skips nothing else)
        g._no_cluster = force
        r0 = GF.deform_backward(g, states, gx, dim, Mu, tau, want_gtau=True)
        r1 = GF.deform_backward(g, states, gx, dim, Mu, tau, want_gtau=True, du=du0)
        assert torch.equal(r0[0], r1[0]) and torch.equal(r0[1], r1[1])
        assert r1[3].shape == du0.shape and torch.isfinite(r1[3]).all()
    g._no_cluster = False


def test_cnn_backward_with_global_gradient_planes(monkeypatch):
    """64x64 grid (gradient planes beyond shared memory) against the fp64 oracle; on a grid that fits, the global-plane
    path (GAD_CNN_GRAD_GLOBAL=1) gives the same bits as the shared-memory one."""
    from g_adaptivity_b200.feature_extractors import GlobalFeatureExtractorCNN
    torch.manual_seed(0)
    for n, B in ((64, 3), (30, 4)):
        m = GlobalFeatureExtractorCNN(1, 8, 8, dim=2, num_layers=4).cuda()
        u = torch.randn(B, 1, n, n)
        cot = torch.randn(B, 8)
        feats = m(u.cuda())
        (feats * cot.cuda()).sum().backward()
        got = {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters()}
        ws = [c.weight.detach().cpu().double().requires_grad_() for c in m.convs]
        bs = [c.bias.detach().cpu().double().requires_grad_() for c in m.convs]
        ref = cnn_oracle.cnn_features(u.double(), ws, bs)
        assert (feats.detach().cpu().double() - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()
        (ref * cot.double()).sum().backward()
        refg = {}
        for l in range(len(m.convs)):
            refg[f"convs.{l}.weight"], refg[f"convs.{l}.bias"] = ws[l].grad, bs[l].grad
        gs = max(g.abs().max().item() for g in refg.values())
        for k, g in refg.items():
            err = (got[k].double() - g).abs().max().item()
            assert err <= 1e-4 * max(g.abs().max().item(), 1e-2 * gs), (n, k, err)
        if n == 30:
            m.zero_grad(set_to_none=True)
            monkeypatch.setenv("GAD_CNN_GRAD_GLOBAL", "1")
            (m(u.cuda()) * cot.cuda()).sum().backward()
            monkeypatch.delenv("GAD_CNN_GRAD_GLOBAL")
            for k, p in m.named_parameters():
                assert torch.equal(p.grad.cpu(), got[k]), k


def test_cnn_backward_1d_long_meshes():
    """1-D meshes of 4000 nodes: the gradient planes live in the workspace too."""
    from g_adaptivity_b200.feature_extractors import GlobalFeatureExtractorCNN
    torch.manual_seed(1)
    m = GlobalFeatureExtractorCNN(1, 8, 8, dim=1, num_layers=4).cuda()
    u, cot = torch.randn(3, 1, 4000), torch.randn(3, 8)
    (m(u.cuda()) * cot.cuda()).sum().backward()
    ws = [c.weight.detach().cpu().double().requires_grad_() for c in m.convs]
    bs = [c.bias.detach().cpu().double().requires_grad_() for c in m.convs]
    (cnn_oracle.cnn_features(u.double(), ws, bs) * cot.double()).sum().backward()
    refg = [t.grad for pair in zip(ws, bs) for t in pair]
    got = [t.grad.cpu() for c in m.convs for t in (c.weight, c.bias)]
    gs = max(g.abs().max().item() for g in refg)
    for a, g in zip(got, refg):
        assert (a.double() - g).abs().max().item() <= 1e-4 * max(g.abs().max().item(), 1e-2 * gs)


@pytest.mark.parametrize("route", ["cluster", "stream", "rk4_stream"])
def test_backward_is_deterministic(route, env):
    over, extra, envd = FU, {}, {"GAD_FWD_POLICY": "cluster"}
    if route == "stream":
        extra, envd = {"gad_no_cluster": True}, {"GAD_FWD_POLICY": "stream"}
    elif route == "rk4_stream":
        over = dict(FU, ode_method="rk4", num_layers=2)
    env(envd)
    _, o1, g1, _ = _run_module((64, 64), 3, over, extra, seed=5)
    _, o2, g2, _ = _run_module((64, 64), 3, over, extra, seed=5)
    assert torch.equal(o1, o2)
    assert g1.keys() == g2.keys()
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k


def test_csr_routes_still_refuse_du():
    from test_gpu_parity import cuda_model
    md = (64, 64)
    opt = synth.default_opt(md, **FU)
    model = cuda_model(_dataset(md), opt, None, gad_no_cluster=True, gad_no_wide=True)
    with pytest.raises(NotImplementedError):
        model(synth.make_batch(md, 2, seed=1))
