"""Global CNN features, gnn_normalize and the learnable temperature through `conv.stored_alpha` and
`GNN.inference_session`.

* stored_alpha of a global-feature model: the CSR read-out with the per-mesh bias offset (gad_conv_alpha_du) against
  the reference's fixtures (tests/golden_glob) and, in 2-D, against the fp64 oracle on every layer and route;
* a session replay equals `model(data)` under no_grad bit for bit, for each option alone and combined, on the
  mesh-resident, cluster and streaming routes, in 1-D and 2-D, across replays with new f / uu;
* `refresh_weights()` is the only way new CNN, Wq / Wk and temperature values reach the replays;
* keeping the alpha source changes no coordinate and no gradient (gad_store_alpha=False is the graph policy global-feature
  models had before they stored alpha)."""
from __future__ import annotations

import copy

import pytest
import torch
import torch.nn.functional as F

import gad_testutil as util
from g_adaptivity_b200 import synth
from oracle import gnn_oracle
from test_glob_features import NAMES, _dataset, _load
from test_gpu_parity import cuda_model

pytestmark = pytest.mark.gpu

FU = {"gnn_inc_glob_feat_f": True, "gnn_inc_glob_feat_uu": True}


@pytest.fixture
def env(monkeypatch):
    def set_env(d):
        for k, v in d.items():
            monkeypatch.setenv(k, v)
    return set_env


def _to64(data):
    d64 = data.clone()
    for k in d64.keys():
        v = getattr(d64, k)
        if torch.is_tensor(v) and v.dtype == torch.float32:
            setattr(d64, k, v.double())
    return d64


def _state_dict(ds, opt):
    """Seeded oracle parameters; learnable temperatures set apart from 1 and from each other."""
    torch.manual_seed(42)
    sd = gnn_oracle.GNNRef(ds, copy.deepcopy(opt)).state_dict()
    for l, k in enumerate(k for k in sd if k.endswith("sm_temp_a")):
        sd[k] = torch.full_like(sd[k], 1.5 + 0.5 * l)
    return sd


# routes: mesh dims, meshes, module extras, environment, tiled graph expected
ROUTES = {
    "tiles_2d": ((12, 12), 4, {}, {}, True),
    "tiles_1d": ((30,), 4, {}, {}, True),
    "cluster_2d": ((64, 64), 2, {}, {"GAD_FWD_POLICY": "cluster"}, False),
    "stream_2d": ((64, 64), 2, {"gad_no_cluster": True}, {"GAD_FWD_POLICY": "stream"}, False),
    "force_stream_1d": ((30,), 4, {"gad_force_stream": True}, {}, True),
    "large_1d": ((4000,), 2, {}, {}, False),
    # dataset on one mesh: graphs that read no attention weights take the shared-topology form (one ELL table for
    # all tiles), the others the general graph -- the two must give the same bits
    "shared_topology_2d": ((12, 12), 4, {"gad_shared_topology": True}, {}, True),
    "shared_topology_1d": ((30,), 4, {"gad_shared_topology": True}, {}, True),
}


# --------------------------------------------------------------------------------------
# stored_alpha with global features
# --------------------------------------------------------------------------------------
@pytest.mark.parametrize("force_stream", [False, True])
@pytest.mark.parametrize("grad", [False, True])
@pytest.mark.parametrize("name", NAMES)
def test_stored_alpha_matches_reference_fixture(name, grad, force_stream):
    fx = _load(name)
    opt, data, md = util.fixture_opt(fx), util.fixture_batch(fx), fx["mesh_dims_list"][0]
    model = cuda_model(_dataset(md), opt, fx["state_dict"], gad_force_stream=force_stream)
    assert model.n_glob_used > 0
    with torch.set_grad_enabled(grad):
        model(data)
    conv = model.conv_layers[-1]
    assert torch.equal(conv.stored_ei.cpu(), fx["edge_index_filtered"])
    alpha = conv.stored_alpha.cpu()
    assert alpha.shape == fx["alpha_last"].shape
    assert (alpha - fx["alpha_last"]).abs().max().item() <= 2e-5


ALPHA_CASES = {
    # id: route, model options
    "rk4_learnable_a": ("tiles_2d", dict(FU, share_conv=False, num_layers=3, ode_method="rk4",
                                         softmax_temp_type="learnable_a")),
    "cluster": ("cluster_2d", dict(FU, share_conv=False, num_layers=3, softmax_temp_type="learnable_a")),
    "stream": ("stream_2d", dict(FU, share_conv=False, num_layers=3)),
    "force_stream": ("tiles_2d", dict(FU, share_conv=False, num_layers=3)),
}


@pytest.mark.parametrize("case", list(ALPHA_CASES))
def test_stored_alpha_matches_oracle_2d(case, env):
    """Every layer's stored_alpha against the fp64 oracle's attention at that layer's input state (with RK4 that is
    the state the step starts from: the read-out does not keep the stage inputs)."""
    route, over = ALPHA_CASES[case]
    md, B, extra, envd, tiled = ROUTES[route]
    if case == "force_stream":
        extra = {"gad_force_stream": True}
    env(envd)
    opt = synth.default_opt(md, **over)
    ds = _dataset(md)
    data = synth.make_batch(md, B, seed=9)
    sd = _state_dict(ds, opt)
    model = cuda_model(ds, opt, sd, **extra)
    ref = gnn_oracle.GNNRef(ds, copy.deepcopy(opt))
    ref.load_state_dict(sd)
    ref = ref.double()
    with torch.no_grad():
        _, states, ei = ref(_to64(data), return_states=True)
        want = []
        for l, layer in enumerate(ref.conv_layers):
            layer(states[l], ei, None, None)
            want.append(layer.stored_alpha.float())
    for grad in (False, True):
        with torch.set_grad_enabled(grad):
            model(data)
        assert (model.last_graph.tile_ptr is not None) == tiled
        for l, conv in enumerate(model.conv_layers):
            assert torch.equal(conv.stored_ei.cpu(), ei)
            err = (conv.stored_alpha.cpu() - want[l]).abs().max().item()
            assert err <= 2e-5, (grad, l, err)


# --------------------------------------------------------------------------------------
# InferenceSession
# --------------------------------------------------------------------------------------
OPTIONS = {
    "glob": FU,
    "glob_uu_without_feat_uu": {"gnn_inc_glob_feat_uu": True, "gnn_inc_feat_uu": False},
    "normalize": {"gnn_normalize": True},
    "learnable_a": {"softmax_temp_type": "learnable_a", "share_conv": False, "num_layers": 3},
    "all": dict(FU, gnn_normalize=True, softmax_temp_type="learnable_a", share_conv=False, num_layers=3),
    "all_rk4": dict(FU, gnn_normalize=True, softmax_temp_type="learnable_a", ode_method="rk4", num_layers=2),
}


def _session_case(route, over):
    md, B, extra, envd, tiled = ROUTES[route]
    opt = synth.default_opt(md, **over)
    ds = _dataset(md)
    model = cuda_model(ds, opt, _state_dict(ds, opt), **extra)
    model.eval()
    return model, synth.make_batch(md, B, seed=5), envd, tiled


def _new_inputs(data, k):
    g = torch.Generator().manual_seed(100 + k)
    f = data.f_tensor * (1.0 + 0.3 * torch.rand(data.f_tensor.shape, generator=g))
    uu = data.uu_tensor * (1.0 + 0.3 * torch.rand(data.uu_tensor.shape, generator=g)) + 0.05 * k
    return f, uu


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("option", list(OPTIONS))
def test_session_replay_equals_module(option, route, env):
    model, data, envd, tiled = _session_case(route, OPTIONS[option])
    env(envd)
    sess = model.inference_session(data)
    assert (sess.graph.tile_ptr is not None) == tiled
    assert getattr(sess.graph, "uniform", False) == route.startswith("shared_topology")
    with torch.no_grad():
        assert torch.equal(sess().clone(), model(data))
        for k in range(3):
            f, uu = _new_inputs(data, k)
            got = sess(f=f.cuda(), uu=uu.cuda()).clone()
            data.f_tensor, data.uu_tensor = f, uu
            want = model(data)
            assert torch.equal(got, want), k
    if OPTIONS[option].get("gnn_inc_glob_feat_f") or OPTIONS[option].get("gnn_inc_glob_feat_uu"):
        assert model.n_glob_used > 0 and sess.cnns


@pytest.mark.parametrize("route", ["tiles_2d", "cluster_2d", "large_1d", "shared_topology_2d"])
def test_session_reads_parameters_on_refresh_only(route, env):
    model, data, envd, _ = _session_case(route, OPTIONS["all"])
    env(envd)
    sess = model.inference_session(data)
    with torch.no_grad():
        before = sess().clone()
        assert torch.equal(before, model(data))
        for name in ("global_feature_extractor_cnn_f", "global_feature_extractor_cnn_uu"):
            getattr(model, name).convs[0].weight.mul_(1.25)
        for conv in model.conv_layers:
            conv.lin_query.weight.add_(0.05)
            conv.lin_key.weight.mul_(0.9)
            conv.sm_temp_a.mul_(1.3)
        after = model(data)
        assert not torch.equal(after, before)
        assert torch.equal(sess().clone(), before)          # nothing leaks in before refresh_weights()
        sess.refresh_weights()
        assert torch.equal(sess().clone(), after)
        assert torch.equal(sess().clone(), model(data))


def test_session_still_refuses_du_on_the_csr_kernels():
    """A global-feature session on a graph only the CSR streaming kernels serve raises, as the module does."""
    md = (64, 64)
    opt = synth.default_opt(md, **FU)
    model = cuda_model(_dataset(md), opt, None, gad_no_cluster=True, gad_no_wide=True)
    with pytest.raises(NotImplementedError):
        model.inference_session(synth.make_batch(md, 2, seed=1))


# --------------------------------------------------------------------------------------
# keeping the alpha source changes nothing the model computes
# --------------------------------------------------------------------------------------
def _train_call(route, over, store):
    md, B, extra, envd, _ = ROUTES[route]
    opt = synth.default_opt(md, **over)
    ds = _dataset(md)
    model = cuda_model(ds, opt, _state_dict(ds, opt), gad_store_alpha=store, **extra)
    model.train()
    data = synth.make_batch(md, B, seed=7)
    out = model(data)
    F.l1_loss(out, data.x_phys.cuda().reshape(out.shape)).backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    with torch.no_grad():
        inf = model(data)
    return model, out.detach(), grads, inf


@pytest.mark.parametrize("option", ["glob", "all"])
@pytest.mark.parametrize("route", list(ROUTES))
def test_alpha_source_leaves_coordinates_and_gradients_unchanged(route, option, env):
    env(ROUTES[route][3])
    over = OPTIONS[option] if option == "glob" else dict(FU, softmax_temp_type="learnable_a", share_conv=False,
                                                         num_layers=3)
    m0, o0, g0, i0 = _train_call(route, over, False)
    m1, o1, g1, i1 = _train_call(route, over, True)
    assert m0.conv_layers[-1].stored_alpha is None and m1.conv_layers[-1].stored_alpha is not None
    if route.startswith("shared_topology"):
        assert getattr(m0.last_graph, "uniform", False) and not getattr(m1.last_graph, "uniform", False)
    assert torch.equal(o0, o1) and torch.equal(i0, i1)
    assert g0.keys() == g1.keys() and any("global_feature" in n for n in g0)
    for n in g0:
        assert torch.equal(g0[n], g1[n]), n
