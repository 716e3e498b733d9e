"""Drop-in `GNN(dataset, opt)` for the g-adaptivity mesh deformer, on sm_100a kernels.

Same constructor reads, `forward(data)` return, parameter names / `state_dict` layout and side
attributes (`end_MLmodel`, `epoch`, `plot_evol_flag`, `conv_layers[i].stored_ei/.stored_alpha`)
as `src/GNN.py:144-306`, so it can stand under `run_GNN.get_model` / `run_pipeline.main`
unchanged.  What differs is underneath:

* the graph prologue of every call (`src/GNN.py:206-223`) runs once on the GPU and is cached
  (`graph.MeshGraph`, K0), found again by tensor identity or by a device content fingerprint when the
  loader hands over a fresh `Batch`;
* feature concat + identity encoder (:225-239, :270), the per-layer Python loop
  `x = x + time_step * layer(x, edge_index)` (:273-296) and the decoder slice (:298-299) are ONE launch
  (`gad_deform_fwd_ell_raw` on meshes that fit a CTA, `gad_deform_fwd_cluster` on larger ones; the
  streaming kernels otherwise), with the folded weights cached per parameter version; autograd's
  op-by-op backward is one hand-written launch plus the reduction;
* `loss_type='pde_loss'` appends the batched differentiable FEM solve (1-D: `fem1d.py`, 2-D: `fem2d.py`, one
  launch for the whole batch instead of the per-mesh Python loop) and returns `(coeffs, x_phys, sol)` as
  `src/GNN.py:307-342` does;
* `inference_session(data)` replays the call as a CUDA graph for roll-outs.

Options the reference supports but this path does not (see SURVEY 8a) raise
`NotImplementedError`; nothing silently falls back to PyTorch, and a non-CUDA device raises.
"""
from __future__ import annotations

import copy
import time
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from . import functional as GF
from .GRAND_plus import GRAND_conv, GRAND_plusConv, inv_temperature
from .feature_extractors import GlobalFeatureExtractorCNN
from .graph import GraphCache, MeshGraph, corner_loops
from .params import get_arg_list


def get_nonlin(nonlin_type):
    table = {"relu": nn.ReLU, "elu": nn.ELU, "selu": nn.SELU, "tanh": nn.Tanh, "sigmoid": nn.Sigmoid,
             "leaky_relu": nn.LeakyReLU, "identity": nn.Identity}
    if nonlin_type not in table:
        raise NotImplementedError(nonlin_type)
    return table[nonlin_type]()


def get_enc(opt, in_dim, out_dim, hid_dim=None, nonlin_type="relu"):
    """`opt['enc'] == 'identity'`: a frozen 0/1 Linear that zero-pads (out >= in) or truncates the
    features (`src/GNN.py:75-90`).  The other encoders crash in the reference (`get_dec` returns
    None for them, :101-105,298) and are rejected here."""
    if opt["enc"] != "identity":
        raise NotImplementedError(f"enc={opt['enc']!r}: only the identity encoder works in the reference")
    lin = nn.Linear(in_dim, out_dim, bias=False)
    k = min(in_dim, out_dim)
    w = torch.zeros(out_dim, in_dim)
    w[:k, :k] = torch.eye(k)
    lin.weight.data = w
    lin.weight.requires_grad = False
    return lin


def get_dec(opt, in_dim, out_dim, hid_dim=None, nonlin_type="relu"):
    if opt["enc"] == "identity":
        return nn.Identity()
    return None


def get_conv(opt, conv_type, in_dim, out_dim, feat_dim=None):
    if conv_type == "GRAND":
        return GRAND_conv(opt, in_dim, out_dim, heads=1)
    if conv_type == "GRAND_plus":
        return GRAND_plusConv(opt, in_dim, out_dim, global_feat_dim=feat_dim, heads=1, concat=False, beta=False,
                              dropout=0.0, edge_dim=None, bias=False, root_weight=False)
    raise NotImplementedError(
        f"conv_type={conv_type!r}: the B200 deformer path implements GRAND_plus and GRAND (north_star); "
        "GCN / GAT / TRANS / GAT_plus are out of scope")


def build_conv_list(opt):
    shared = None
    if opt["share_conv"]:
        shared = get_conv(opt, opt["conv_type"], opt["hidden_dim"], opt["hidden_dim"], opt["global_feat_dim"])
    layers = []
    for _ in range(opt["num_layers"]):
        layers.append(shared if shared is not None else
                      get_conv(opt, opt["conv_type"], opt["hidden_dim"], opt["hidden_dim"], opt["global_feat_dim"]))
    return nn.ModuleList(layers)


class GNN(nn.Module):
    def __init__(self, dataset, opt):
        super().__init__()
        self.dataset = dataset
        self.opt = opt
        self.dim = dataset.num_x_comp_features
        self.mesh_dims = get_arg_list(opt["mesh_dims"])
        self.in_dims = [self.dim]
        if opt["gnn_inc_feat_f"]:
            self.in_dims += [1]
        if opt["gnn_inc_feat_uu"]:
            self.in_dims += [1]
        z_dim = sum(self.in_dims)                      # node-varying input channels: x_comp [, f] [, uu]
        glob_f, glob_uu = bool(opt["gnn_inc_glob_feat_f"]), bool(opt["gnn_inc_glob_feat_uu"])
        if glob_f:
            self.in_dims += [opt["global_feat_dim"]]
        if glob_uu:
            self.in_dims += [opt["global_feat_dim"]]
        opt["hidden_dims_list"] = self.in_dims

        in_dim = sum(self.in_dims)
        hid_dim = opt["hidden_dim"]
        self.enc = get_enc(opt, in_dim, hid_dim, nonlin_type=opt["non_lin"])
        self.conv_layers = build_conv_list(opt)
        self.non_lin = get_nonlin(opt["non_lin"])
        self.dec = get_dec(opt, hid_dim, self.dim, nonlin_type=opt["non_lin"])
        # global CNN features (src/GNN.py:172-177): created after the conv layers, f before uu, as the reference does
        # (same parameter order, same random stream)
        if glob_f:
            self.global_out_dim = opt["global_feat_dim"]
            self.global_feature_extractor_cnn_f = GlobalFeatureExtractorCNN(1, hid_dim, self.global_out_dim, dim=self.dim)
        if glob_uu:
            self.global_out_dim = opt["global_feat_dim"]
            self.global_feature_extractor_cnn_uu = GlobalFeatureExtractorCNN(1, hid_dim, self.global_out_dim, dim=self.dim)
        # The identity encoder keeps the first hidden_dim input channels (src/GNN.py:84-90).  Of the global channels that
        # survive, every mesh carries a CONSTANT vector: the state rows stay dim + f + uu wide and the global part
        # enters the kernels as a per-mesh offset of the folded bias (include/gadapt.h: `du`).
        self.z_dim = z_dim
        self.n_glob_used = max(0, min(hid_dim, in_dim) - z_dim) if (glob_f or glob_uu) else 0
        if opt["learn_step"]:
            self.steps = nn.ParameterList([nn.Parameter(torch.tensor([opt["time_step"]]))
                                           for _ in range(opt["num_layers"])])
        if self.dim == 1:
            self.quad_points = torch.linspace(0, 1, opt["eval_quad_points"])
        elif self.dim == 2:
            x0 = torch.linspace(0, 1, opt["eval_quad_points"])
            X, Y = torch.meshgrid(x0, x0, indexing="ij")
            self.quad_points = [X, Y]

        self._validate(opt)
        self.live, self.CE = GF.live_channels(z_dim, hid_dim)
        self.inv_temp = inv_temperature(opt) if opt["conv_type"] == "GRAND_plus" else 1.0
        self._graphs = GraphCache(capacity=int(opt.get("gad_graph_cache", 8)))
        self._tau_const = None
        self.end_MLmodel = None
        self.last_graph = None

    # ------------------------------------------------------------------------------------
    def _validate(self, opt):
        if not opt["residual"]:
            raise NotImplementedError("residual=False replaces x by F(x) and is only meaningful for non-GRAND convs")
        if opt.get("dropout", 0.0) != 0.0:
            raise NotImplementedError("dropout > 0 is off the deformer hot path")
        if opt["conv_type"] == "GRAND" and opt["non_lin"] != "identity":
            raise NotImplementedError("GRAND with a non-identity non_lin (src/GNN.py:286) is not implemented")
        if opt.get("ode_method", "euler") not in GF.METHODS:
            raise ValueError(f"ode_method must be one of {sorted(GF.METHODS)}")
        if opt["loss_type"] == "pde_loss" and opt.get("data_type") == "randg_mix":
            raise NotImplementedError(
                "loss_type='pde_loss' with data_type='randg_mix' solves on a different Firedrake mesh per sample "
                "(data.mesh[b], src/GNN.py:316-318): the batched FEM kernels share one triangulation per batch")
        if opt["loss_type"] not in ("mesh_loss", "modular", "pde_loss"):
            raise NotImplementedError(f"loss_type={opt['loss_type']!r} is not implemented")

    def _device(self):
        dev = torch.device(self.opt["device"])
        if dev.type != "cuda":
            raise RuntimeError(
                f"opt['device']={self.opt['device']!r}: the B200 deformer has no CPU path (no fallback by design); "
                "use the oracle in oracle/ for CPU reference numbers")
        return dev

    @staticmethod
    def _mesh_sizes(data) -> List[int]:
        if getattr(data, "mesh_sizes", None) is not None:
            return list(data.mesh_sizes)
        if getattr(data, "ptr", None) is not None:     # PyG Batch
            return torch.diff(data.ptr).cpu().tolist()
        return torch.bincount(data.batch).cpu().tolist()

    def _graph(self, data, dev, allow_uniform: bool = False, tile_nodes: Optional[int] = None) -> MeshGraph:
        """The cached result of the graph prologue (src/GNN.py:206-223) for this batch.  `allow_uniform`: the caller
        only runs the mesh-resident ELL kernels and does not read attention weights, so with
        `opt['gad_shared_topology']` (dataset on one mesh) the graph may be the shared-topology form, built for one
        tile (`MeshGraph.build_uniform`)."""
        opt = self.opt
        uniform_ok = bool(allow_uniform and opt.get("gad_shared_topology", False)
                          and not any(opt.get(k, False) for k in ("gad_no_ell", "gad_force_stream", "gad_no_fused_train")))
        tile_target = tile_nodes if tile_nodes is not None else opt.get("gad_tile_nodes")
        flags = (bool(opt["fix_boundary"]), bool(opt["self_loops"]), self.CE, str(dev), tile_target,
                 bool(opt.get("gad_no_ell", False)), bool(opt.get("gad_no_wide", False)), bool(opt.get("gad_no_cluster", False)),
                 uniform_ok)
        key = GraphCache.key_of(data, flags)
        g = self._graphs.get(key)
        if g is not None:
            return g
        # Identity miss (a fresh Batch from the loader).  Datasets on one shared mesh: shapes + host samples
        skey = None
        if opt.get("gad_shared_topology", False):
            skey = GraphCache.shared_key_of(data, flags)
            g = self._graphs.get(skey)
            if g is not None:
                self._graphs.shared_hits = getattr(self._graphs, "shared_hits", 0) + 1
                return g
        if uniform_ok:
            g = MeshGraph.build_uniform(data, self._mesh_sizes(data), self.dim, opt["mesh_dims"], bool(opt["fix_boundary"]),
                                        bool(opt["self_loops"]), dev, ce=self.CE, tile_target=tile_target)
            if g is not None:
                keep = (data.edge_index, data.batch) + tuple(getattr(data, n, None) for n in GraphCache.TOPOLOGY_FIELDS)
                self._graphs.put(key, g, keep)
                self._graphs._d[skey] = g
                return g
        # otherwise look the topology up by CONTENT before building
        ckey, dev_copies = None, {}
        if opt.get("gad_content_cache", True):
            ckey, dev_copies = GraphCache.content_key_of(data, flags, dev, use_masks=bool(opt["fix_boundary"]))
            g = self._graphs.get(ckey)
            if g is not None:
                self._graphs.misses_identity = getattr(self._graphs, "misses_identity", 0) + 1
                self._graphs.alias(key, g, tuple(getattr(data, n, None) for n in GraphCache.TOPOLOGY_FIELDS))
                return g
        sizes = self._mesh_sizes(data)
        N = int(data.x_comp.shape[0])
        masks, loops = (), None
        if opt["fix_boundary"]:
            masks = tuple(dev_copies.get(n, getattr(data, n)) for n in
                          ("to_boundary_edge_mask", "to_corner_nodes_mask", "diff_boundary_edges_mask"))
            loops = corner_loops(data, self.dim, opt["mesh_dims"], sizes)
        g = MeshGraph.build(dev_copies.get("edge_index", data.edge_index), N, masks=masks, extra_loops=loops,
                            self_loops=bool(opt["self_loops"]),
                            mesh_sizes=sizes, device=dev, ce=self.CE, tile_target=tile_target,
                            use_ell=not opt.get("gad_no_ell", False))
        if opt.get("gad_no_wide", False):
            g._wide_tried = True          # keep the CSR streaming kernels (csrc/stream_kernels.cu)
        if opt.get("gad_no_cluster", False):
            g._no_cluster = True          # keep the streaming kernels for meshes beyond one CTA
        keep = (data.edge_index, data.batch) + tuple(getattr(data, n, None) for n in GraphCache.TOPOLOGY_FIELDS)
        self._graphs.put(key, g, keep)
        if ckey is not None:
            self._graphs._d[ckey] = g
        if skey is not None:
            self._graphs._d[skey] = g
        return g

    def _plan_graph(self, data, dev, allow_uniform: bool) -> MeshGraph:
        """The graph a call runs on (the module and InferenceSession both plan here).  With global CNN features the bias
        offset is per tile, so tiles hold one mesh each; a mesh too large for the mesh-resident ELL kernels gets the graph
        a model without global features builds, which runs on the cluster / streaming kernels (they take the offset per
        mesh), not on CSR tiles."""
        tile_nodes = None
        if self.n_glob_used:
            sizes = self._mesh_sizes(data)
            if any(n != sizes[0] for n in sizes):
                raise NotImplementedError("global CNN features need meshes of equal size in a batch")
            tile_nodes = int(sizes[0])
        graph = self._graph(data, dev, allow_uniform=allow_uniform, tile_nodes=tile_nodes)
        if tile_nodes is not None and graph.tile_ptr is not None and not GF.use_ell(graph, self.CE):
            graph = self._graph(data, dev, allow_uniform=allow_uniform)
        return graph

    def _softmax_temps(self) -> Optional[torch.Tensor]:
        """[Lw] learnable temperatures of `softmax_temp_type='learnable_a'` (src/GRAND_plus.py:152-154,328-329), or None."""
        if self.opt.get("softmax_temp_type") != "learnable_a":
            return None
        convs = [self.conv_layers[0]] if self.opt["share_conv"] else list(self.conv_layers)
        return torch.cat([c.sm_temp_a.reshape(1) for c in convs])

    def _folded_weights(self, dev):
        """(M, u) of the current Linear parameters (csrc/weights.cu), cached until a parameter changes:
        keyed on storage and version counter of every parameter plus `_param_epoch`, which the
        trainer bumps because its kernels update the parameters without touching the counters."""
        convs = [self.conv_layers[0]] if self.opt["share_conv"] else list(self.conv_layers)
        ps = [p for c in convs for p in (c.lin_query.weight, c.lin_query.bias, c.lin_key.weight)]
        key = (tuple((p.data_ptr(), p._version) for p in ps), getattr(self, "_param_epoch", 0), self.inv_temp, dev)
        if getattr(self, "_mu_key", None) != key:
            Wq, bq, Wk, _ = self._weights()
            self._mu = GF.prepare_weights(Wq.detach(), bq.detach(), Wk.detach(), self.CE, self.inv_temp)
            self._mu_key = key
        return self._mu

    def _weights(self):
        convs = [self.conv_layers[0]] if self.opt["share_conv"] else list(self.conv_layers)
        if len(convs) == 1:      # views: no kernels, no copies
            c = convs[0]
            return (c.lin_query.weight.unsqueeze(0), c.lin_query.bias.unsqueeze(0), c.lin_key.weight.unsqueeze(0),
                    c.lin_key.bias.unsqueeze(0))
        Wq = torch.stack([c.lin_query.weight for c in convs])
        bq = torch.stack([c.lin_query.bias for c in convs])
        Wk = torch.stack([c.lin_key.weight for c in convs])
        bk = torch.stack([c.lin_key.bias for c in convs])
        return Wq, bq, Wk, bk

    def _tau(self, dev):
        if self.opt["learn_step"]:
            return torch.cat([s.reshape(1) for s in self.steps])
        if self._tau_const is None or self._tau_const.device != dev:
            self._tau_const = torch.full((self.opt["num_layers"],), float(self.opt["time_step"]),
                                         dtype=torch.float32, device=dev)
        return self._tau_const

    # ------------------------------------------------------------------------------------
    def forward(self, data):
        opt = self.opt
        dev = self._device()
        keep_alpha = isinstance(opt.get("show_mesh_evol_plots"), bool) or opt["conv_type"] == "GRAND"
        keep_alpha = keep_alpha and bool(opt.get("gad_store_alpha", True))
        graph = self._plan_graph(data, dev, allow_uniform=not keep_alpha)
        x_comp = data.x_comp.to(dev, non_blocking=True)
        f = data.f_tensor.to(dev, non_blocking=True) if opt["gnn_inc_feat_f"] else None
        uu = data.uu_tensor.to(dev, non_blocking=True) if opt["gnn_inc_feat_uu"] else None
        f_scale = uu_scale = None
        if opt["gnn_normalize"]:                       # f / torch.max(f): signed batch-wide max (GNN.py:231-237)
            f_scale = torch.max(f).reshape(1).float() if f is not None else None
            uu_scale = torch.max(uu).reshape(1).float() if uu is not None else None
        if x_comp.dim() == 1:
            x_comp = x_comp.unsqueeze(-1)
        tau = self._tau(dev)
        Mu_in = self._folded_weights(dev)
        aux = {"keep_states": keep_alpha, "Mu_in": Mu_in}
        du = self._global_bias_offsets(data, graph, f, uu, f_scale, uu_scale, dev) if self.n_glob_used else None
        temp = self._softmax_temps()                            # per weight set
        if temp is not None and du is not None:
            du = du / temp.reshape(1, -1, 1)                     # the bias offset is a logit term too
        method = GF.METHODS[opt.get("ode_method", "euler")]
        force_stream = bool(opt.get("gad_force_stream", False))
        if not torch.is_grad_enabled():
            # inference: no autograd node; on mesh-resident graphs the whole call is one kernel launch
            N = x_comp.shape[0]
            L = int(tau.numel())
            states = torch.empty((L, N, self.CE), dtype=torch.float32, device=dev) if keep_alpha else None
            Mu_eff = Mu_in if temp is None else (Mu_in / temp.detach().float().reshape(-1, 1)).contiguous()
            x_phys = GF.deform_forward_raw(graph, x_comp, f, uu, f_scale, uu_scale, self.dim, self.CE, Mu_eff,
                                           GF._f32(tau.detach().reshape(-1)), method, states=states,
                                           force_stream=force_stream, du=None if du is None else du.detach().contiguous())
            aux["states"], aux["Mu"] = states, Mu_eff
        else:
            Wq, bq, Wk, bk = self._weights()
            x_phys = GF.DeformFunction.apply(
                x_comp, f, uu, f_scale, uu_scale, Wq, bq, Wk, bk, tau, graph, self.dim, self.CE, self.inv_temp,
                method, force_stream, aux, du, temp)
        if keep_alpha and aux.get("states") is not None:
            states, Mu = aux["states"], aux["Mu"]
            du_a = None if du is None else du.detach()          # the offset the deformer ran with (temperature included)
            L = opt["num_layers"]
            if opt["share_conv"]:
                self.conv_layers[0]._set_alpha_source(graph, states[L - 1], Mu[0:1], None if du_a is None else du_a[:, 0])
            else:
                for l, conv in enumerate(self.conv_layers):
                    conv._set_alpha_source(graph, states[l], Mu[l:l + 1], None if du_a is None else du_a[:, l])
        object.__setattr__(self, "last_graph", graph)      # plain attributes: nn.Module.__setattr__ costs 2 us each
        # `end_MLmodel` is read by the reference's evaluation code as the end of the model's run time
        # (src/utils_eval.py:193-201): in eval mode the stamp is taken after the stream has drained; the training
        # loop stays asynchronous.  opt['gad_sync_timestamp'] overrides either way.
        if opt.get("gad_sync_timestamp", not self.training):
            torch.cuda.current_stream(dev).synchronize()
        object.__setattr__(self, "end_MLmodel", time.time())
        if opt["loss_type"] == "pde_loss" and self.dim == 2:
            return self._pde_tail_2d(data, graph, x_phys, dev)
        if opt["loss_type"] == "pde_loss":
            # src/GNN.py:307-342 (dim == 1): per mesh torch_FEM_1D on its relocated points -> one batched launch.
            # Returns (coeffs_batched [B*(n-2), 1], x_phys_batched [N], sol_batched [B*Q]) like the reference.
            from . import fem1d
            B, n = self._pde_batch_shape(data, graph, int(x_phys.shape[0]))
            centers, scales = self._pde_gaussians(data, B, dev)
            (quad,), _ = self._pde_eval_points(dev)
            xp = x_phys.squeeze(-1)
            coeffs, sol = fem1d.fem1d_solve(xp, centers, scales, quad, n, int(opt.get("load_quad_points", 101)))
            return coeffs, xp, sol
        return x_phys

    # ------------------------------------------------------------------------------------
    # set-up of loss_type='pde_loss', shared by the module's FEM tail and DeformerTrainer's pde slots
    @staticmethod
    def _pde_batch_shape(data, graph, num_nodes: int):
        """(B, nodes per mesh) of a pde_loss batch; the batched FEM kernels need meshes of one size."""
        B = len(graph.mesh_sizes) if graph.mesh_sizes is not None else int(data.batch.max().item()) + 1
        n = num_nodes // B
        if graph.mesh_sizes is not None and any(m != n for m in graph.mesh_sizes):
            raise NotImplementedError("pde_loss needs meshes of equal size in a batch")
        return B, n

    def _pde_gaussians(self, data, B: int, dev):
        """(centers, scales) of `data.pde_params` as the FEM kernels take them: 1-D fp32 [B, G], 2-D fp64 [B, G, 2].
        The Gaussian parameters of a batch object do not change between epochs: converted once per object (the entry
        keeps the dict alive, so its id cannot be recycled while it is cached)."""
        cache = self.__dict__.setdefault("_pde_cache", {})
        hit = cache.get(id(data.pde_params))
        if hit is None or hit[0] is not data.pde_params or hit[1].shape[0] != B:
            if len(cache) >= 64:
                cache.clear()
            hit = (data.pde_params,) + self._pde_params_to_tensors(data.pde_params, B, dev)
            cache[id(data.pde_params)] = hit
        return hit[1], hit[2]

    def _pde_params_to_tensors(self, pde_params, B: int, dev) -> tuple:
        """`pde_params` -> (centers, scales) in the FEM kernels' layout and precision, uncached."""
        from . import fem1d, fem2d
        to_tensors = fem2d.pde_params_to_tensors if self.dim == 2 else fem1d._pde_params_to_tensors
        return to_tensors(pde_params, B, dev)

    def _pde_eval_points(self, dev):
        """Where the FEM solution is evaluated, and the order the loss reads it in (cached on the device):
        1-D ((quad [Q],), None); 2-D ((X [Q*Q], Y [Q*Q]), order [Q*Q] int64).  2-D `order` is
        argsort(mapping_tensor_fine): `reshape_grid_to_fd_tensor(sol.view(-1).unsqueeze(-1), mapping_tensor_fine)`
        (utils_data.py:143-159) is `sol.view(-1)[order]` for this call shape."""
        ev = self.__dict__.get("_pde_eval")
        if ev is None or ev[0][0].device != dev:
            if self.dim == 2:
                X, Y = self.quad_points
                mapping = getattr(self.dataset, "mapping_tensor_fine", None)
                if mapping is None:
                    raise ValueError("loss_type='pde_loss' on 2-D meshes needs dataset.mapping_tensor_fine (src/GNN.py:333)")
                _, order = torch.sort(torch.as_tensor(mapping).reshape(-1))           # utils_data.py:154
                ev = ((X.reshape(-1).to(dev, torch.float32).contiguous(), Y.reshape(-1).to(dev, torch.float32).contiguous()),
                      order.to(dev))
            else:
                ev = ((self.quad_points.to(dev, torch.float32).contiguous(),), None)
            self.__dict__["_pde_eval"] = ev
        return ev

    # ------------------------------------------------------------------------------------
    def _global_bias_offsets(self, data, graph, f, uu, f_scale, uu_scale, dev):
        """Global CNN features (src/GNN.py:242-268) as the per-mesh offset of the folded bias the kernels take.

        The reference appends g_b = [CNN_f(f grid) | CNN_uu(uu grid)] of mesh b to the features of each of its nodes;
        the identity encoder keeps the first `hidden_dim` channels.  Constant channels stay constant under
        x <- x + tau (A x - x), and in the logit  x_i^T M x_j + u^T x_j  (M = c Wq^T Wk) every term they enter is
        constant over the in-edges of i -- it cancels in the softmax -- except  g^T M[z:, :z] z_j.  So the deformer
        sees them as  u_b = u + M[z:z+n_g, :z]^T g_b : du [B, Lw, CE], differentiable with respect to the CNN
        parameters (hand-written backward, csrc/glob_cnn.cu) and to Wq / Wk (a [n_g x z] matrix product per
        weight set, left to autograd)."""
        opt = self.opt
        sizes = self._mesh_sizes(data)
        B, N1 = len(sizes), int(sizes[0])
        gather = self._cnn_grid_map(data, N1, dev)
        if opt["gnn_inc_glob_feat_f"] and f is None:
            f = data.f_tensor.to(dev, non_blocking=True)
        if opt["gnn_inc_glob_feat_uu"] and uu is None:
            uu = data.uu_tensor.to(dev, non_blocking=True)
        Wq, _, Wk, _ = self._weights()
        return self._bias_offsets(B, N1, gather, f, uu, f_scale, uu_scale, Wq, Wk,
                                  getattr(self, "global_feature_extractor_cnn_f", None),
                                  getattr(self, "global_feature_extractor_cnn_uu", None))

    def _bias_offsets(self, B: int, N1: int, gather, f, uu, f_scale, uu_scale, Wq, Wk, cnn_f, cnn_uu) -> torch.Tensor:
        """du [B, Lw, CE] of `_global_bias_offsets` from device tensors only (no host synchronisation, so that
        InferenceSession can capture it): B meshes of N1 nodes, the CNNs' inputs f / uu [B * N1], the deformer's
        gnn_normalize maxima, Wq / Wk [Lw, C, C] and the two CNN modules (None where the option is off)."""
        opt = self.opt
        lib_c = GF.fold_scale(self.inv_temp, int(opt["hidden_dim"]))
        feats = []
        if opt["gnn_inc_glob_feat_f"]:
            src = f
            if opt["gnn_inc_feat_f"] and f_scale is not None:
                src = src / f_scale                      # the reference normalises f in place before the CNN sees it (:231-233)
            feats.append(cnn_f(src.reshape(B, N1), gather=gather))
        if opt["gnn_inc_glob_feat_uu"]:
            src = uu
            if opt["gnn_inc_feat_uu"] and uu_scale is not None:
                src = src / uu_scale
            feats.append(cnn_uu(src.reshape(B, N1), gather=gather))
        g = torch.cat(feats, dim=1)[:, :self.n_glob_used]                 # what the encoder's truncation keeps
        z0, z1 = self.z_dim, self.z_dim + self.n_glob_used
        M = lib_c * torch.matmul(Wq.transpose(1, 2), Wk)                  # [Lw, C, C], log2-domain scale of the kernels
        du = torch.einsum("bg,lgz->blz", g, M[:, z0:z1, :self.live])      # [B, Lw, live]
        if self.live < self.CE:
            du = torch.nn.functional.pad(du, (0, self.CE - self.live))
        return du.contiguous()

    def _cnn_grid_map(self, data, N1: int, dev) -> torch.Tensor:
        """int32 [N1]: the node of a mesh whose value sits in each cell of the CNN's grid (cached)."""
        opt = self.opt
        gather = self.__dict__.get("_cnn_gather")
        if gather is None or gather.numel() != N1 or gather.device != dev:
            if self.dim == 2:
                mapping = getattr(self.dataset, "mapping_tensor", None)
                if opt.get("data_type") == "randg_mix":
                    mapping = getattr(data, "mapping_tensor", mapping)
                if mapping is None:
                    raise ValueError("global CNN features on 2-D meshes need dataset.mapping_tensor (src/GNN.py:245)")
                n = int(round(N1 ** 0.5))
                # reshape_fd_tensor_to_grid (utils_data.py:125-141): gather by the mapping, reshape [n, n], transpose,
                # flip rows -- as ONE index map applied by the kernel's load: grid[r, c] = u[mapping[c * n + n - 1 - r]]
                r, c = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
                gather = torch.as_tensor(mapping).reshape(-1)[(c * n + (n - 1 - r)).reshape(-1)].to(dev, torch.int32)
            else:
                gather = torch.arange(N1, dtype=torch.int32, device=dev)
            self.__dict__["_cnn_gather"] = gather
        return gather

    def _fem2d_topology(self, dev, num_nodes: int):
        """Triangulation tables of `dataset.mesh` for the batched 2-D FEM kernels, built once per model.
        The reference reads `mesh.coordinates.cell_node_map().values` and `DirichletBC(V, 0, "on_boundary").nodes`
        (difFEM_2d.py:354-356,363); a mesh object that carries `bc_nodes` (synth.SyntheticMesh, or any stand-in)
        is used as is, a Firedrake mesh is asked through Firedrake."""
        from . import fem2d
        topo = self.__dict__.get("_fem2d_topo")
        if topo is not None and topo.N == num_nodes and topo.device == dev:
            return topo
        mesh = getattr(self.dataset, "mesh", None)
        if mesh is None:
            raise ValueError("loss_type='pde_loss' on 2-D meshes needs dataset.mesh (src/GNN.py:321)")
        cells = np.asarray(mesh.coordinates.cell_node_map().values)
        if hasattr(mesh, "bc_nodes"):
            bc = np.asarray(mesh.bc_nodes)
        else:
            from firedrake import DirichletBC, FunctionSpace      # the reference's own route
            bc = np.asarray(DirichletBC(FunctionSpace(mesh, "CG", 1), 0, "on_boundary").nodes)
        topo = fem2d.Fem2DTopology(cells, bc, num_nodes, dev)
        self.__dict__["_fem2d_topo"] = topo
        return topo

    def _pde_tail_2d(self, data, graph, x_phys, dev):
        """src/GNN.py:307-342 with dim == 2: per mesh `torch_FEM_2D` on its relocated points, then the solution on
        the evaluation grid is put into the fine mesh's node order by `reshape_grid_to_fd_tensor(sol.view(-1)
        .unsqueeze(-1), dataset.mapping_tensor_fine)` (utils_data.py:143-159: for this call shape that is
        `sol.view(-1)[argsort(mapping_tensor_fine)]`).  Here: ONE batched launch (csrc/fem2d.cu) + one gather.
        Returns (coeffs [B*n*n, 1], x_phys [B*n*n, 2], sol [B*Q*Q]) like the reference."""
        from . import fem2d
        B, Nm = self._pde_batch_shape(data, graph, int(x_phys.shape[0]))
        topo = self._fem2d_topology(dev, Nm)
        centers, scales = self._pde_gaussians(data, B, dev)
        (ex, ey), order = self._pde_eval_points(dev)
        sol, coeffs, _ = fem2d.fem2d_solve(x_phys.view(B, Nm, 2), topo, centers, scales, ex, ey,
                                           int(self.opt.get("load_quad_points", 101)))
        sol_fd = sol.index_select(1, order)
        return coeffs.reshape(B * Nm, 1), x_phys, sol_fd.reshape(-1)

    def inference_session(self, data) -> "InferenceSession":
        """Replayable deformer call on a fixed topology (extension; the Burgers roll-out of
        src/utils_eval_Burgers.py:269,297 calls the model on the same mesh with a new `uu` every time
        step): static device copies of the inputs, one captured CUDA graph holding the single
        forward launch; `session(uu=...)` refreshes inputs and replays."""
        return InferenceSession(self, data)


class InferenceSession:
    """`GNN.forward(data)` in inference mode as one CUDA-graph replay (see GNN.inference_session).

    The output tensor is static: it is overwritten by the next call.  Parameters are read when the session is created
    (and again by `refresh_weights()`): the folded weights, the step sizes, the learnable temperatures and, with global
    CNN features, the CNN parameters and the Wq / Wk the bias offset is formed from.  What depends on the node inputs
    -- the gnn_normalize maxima, the CNN features with their abs-max scale, the bias offset -- is recomputed inside the
    graph on every replay by the module's own arithmetic, so a replay gives the bits of `model(data)` under no_grad."""

    def __init__(self, model: GNN, data):
        opt = model.opt
        self.model, self.dev = model, model._device()
        dev = self.dev
        self.graph = model._plan_graph(data, dev, allow_uniform=True)
        f32 = dict(dtype=torch.float32, device=dev)
        xc = data.x_comp if data.x_comp.dim() == 2 else data.x_comp.unsqueeze(-1)
        self.x_comp = xc.to(**f32).contiguous().clone()
        glob = model.n_glob_used > 0
        # f / uu are kept when the deformer or a CNN reads them
        need_f = opt["gnn_inc_feat_f"] or (glob and opt["gnn_inc_glob_feat_f"])
        need_uu = opt["gnn_inc_feat_uu"] or (glob and opt["gnn_inc_glob_feat_uu"])
        self.f = data.f_tensor.to(**f32).contiguous().clone() if need_f else None
        self.uu = data.uu_tensor.to(**f32).contiguous().clone() if need_uu else None
        self.tau = GF._f32(model._tau(dev).detach().reshape(-1)).clone()
        temp = model._softmax_temps()
        self.temp = None if temp is None else temp.detach().float().clone()
        self.Mu = self._read_mu()
        self.cnns = None
        if glob:
            sizes = model._mesh_sizes(data)
            self.B, self.N1 = len(sizes), int(sizes[0])
            self.gather = model._cnn_grid_map(data, self.N1, dev)
            Wq, _, Wk, _ = model._weights()
            self.Wq, self.Wk = Wq.detach().clone(), Wk.detach().clone()
            self.cnns = {k: copy.deepcopy(getattr(model, "global_feature_extractor_cnn_" + k)).requires_grad_(False)
                         for k in ("f", "uu") if opt["gnn_inc_glob_feat_" + k]}
        self.method = GF.METHODS[opt.get("ode_method", "euler")]
        self.force_stream = bool(opt.get("gad_force_stream", False))
        self.stream = torch.cuda.Stream(device=dev)
        self.out = None
        with torch.cuda.device(dev), torch.no_grad():
            self.stream.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(self.stream):
                self._call()                       # warm-up: attribute set-up, allocations
            self.stream.synchronize()
            self.cuda_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.cuda_graph, stream=self.stream):
                self.out = self._call()
            torch.cuda.current_stream(dev).wait_stream(self.stream)

    def _read_mu(self) -> torch.Tensor:
        """The folded weights the module's no_grad call runs on: (M, u) / T with a learnable temperature."""
        Mu = self.model._folded_weights(self.dev)
        if self.temp is not None:
            Mu = (Mu / self.temp.reshape(-1, 1)).contiguous()
        return Mu.clone()

    def _call(self):
        m, opt = self.model, self.model.opt
        f = self.f if opt["gnn_inc_feat_f"] else None
        uu = self.uu if opt["gnn_inc_feat_uu"] else None
        f_scale = uu_scale = None
        if opt["gnn_normalize"]:                   # GNN.forward: signed batch-wide max of the current inputs
            f_scale = torch.max(f).reshape(1).float() if f is not None else None
            uu_scale = torch.max(uu).reshape(1).float() if uu is not None else None
        du = None
        if self.cnns is not None:
            du = m._bias_offsets(self.B, self.N1, self.gather, self.f, self.uu, f_scale, uu_scale, self.Wq, self.Wk,
                                 self.cnns.get("f"), self.cnns.get("uu"))
            if self.temp is not None:
                du = du / self.temp.reshape(1, -1, 1)
        return GF.deform_forward_raw(self.graph, self.x_comp, f, uu, f_scale, uu_scale, m.dim, m.CE, self.Mu, self.tau,
                                     self.method, states=None, force_stream=self.force_stream, du=du)

    def refresh_weights(self):
        """Re-read the model's parameters (on the caller's current stream, like the replays)."""
        m = self.model
        with torch.no_grad():
            if self.temp is not None:
                self.temp.copy_(m._softmax_temps())
            self.Mu.copy_(self._read_mu())
            self.tau.copy_(GF._f32(m._tau(self.dev).detach().reshape(-1)))
            if self.cnns is not None:
                Wq, _, Wk, _ = m._weights()
                self.Wq.copy_(Wq)
                self.Wk.copy_(Wk)
                for k, cnn in self.cnns.items():
                    for mine, theirs in zip(cnn.parameters(), getattr(m, "global_feature_extractor_cnn_" + k).parameters()):
                        mine.copy_(theirs)

    def __call__(self, x_comp=None, f=None, uu=None) -> torch.Tensor:
        """Replay with (optionally) new node inputs; returns the static output tensor [N, dim].  The input copies
        and the replay are issued on the CALLER's current stream (a captured graph replays on whatever stream is
        current), so the call is ordered like any other op of that stream and costs no cross-stream events."""
        if x_comp is not None:
            self.x_comp.copy_(x_comp if x_comp.dim() == 2 else x_comp.unsqueeze(-1), non_blocking=True)
        if f is not None and self.f is not None:
            self.f.copy_(f, non_blocking=True)
        if uu is not None and self.uu is not None:
            self.uu.copy_(uu, non_blocking=True)
        self.cuda_graph.replay()
        return self.out
