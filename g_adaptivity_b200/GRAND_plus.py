"""Operator seam: `GRAND_plusConv` / `GRAND_conv` on the sm_100a kernels.

Mirrors the constructor and `forward` surface of `src/GRAND_plus.py:40-343` (GRAND_plusConv) and
`:366-382` (GRAND_conv) for the configuration the deformer builds (`src/GNN.py:115-119`:
heads=1, concat=False, beta=False, dropout=0, edge_dim=None, bias=False, root_weight=False), with
the same parameter names so a reference `state_dict` loads unchanged:
`lin_key.{weight,bias}`, `lin_query.{weight,bias}`, `lin_skip.weight` (constructed, never used --
`root_weight=False` -- exactly as in the reference).

`forward(x, edge_index, ...)` returns `A(x) x - x` (`src/GRAND_plus.py:267`): q/k projection,
edge logits, segment softmax over incoming edges, aggregation and the `- x` in one kernel
(`gad_conv_fwd`), with a hand-written backward (`gad_conv_bwd`).  Inside `GNN.forward` the layers
are not called one by one: the model hands all L layers to the fused integrator instead.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from . import functional as GF
from .graph import GraphCache, MeshGraph

_UNSUPPORTED_TEMP = ("learnable_v",)


def inv_temperature(opt: dict) -> float:
    """`softmax_temp_type == 'fixed'` divides the logits by `softmax_temp` (`src/GRAND_plus.py:326-327`);
    `'learnable_a'` divides them by the layer's learnable scalar `sm_temp_a` (:152-154,328-329), which the model
    applies as a factor on the folded weights (so this returns 1); every other CLI value falls through to the plain
    softmax (:332-333).  `'learnable_v'` applies `Linear(C, H)` to the `[E, H]` logits in the reference (:158,331), a
    shape error there: rejected."""
    t = opt.get("softmax_temp_type")
    if t in _UNSUPPORTED_TEMP:
        raise NotImplementedError(
            f"softmax_temp_type={t!r} is unreachable from the reference CLI and a shape error there "
            "(src/GRAND_plus.py:158,331); not implemented")
    if t == "fixed":
        return 1.0 / float(opt["softmax_temp"])
    return 1.0


class _AlphaSource:
    """Everything needed to materialise `stored_alpha` on demand (it costs an [E] write, so it is
    not produced on every call the way the reference does, `src/GRAND_plus.py:253-256`).  `du` [meshes, CE]: the
    per-mesh bias offset of the layer's weight set (global CNN features), or None."""

    def __init__(self, graph: MeshGraph, x: torch.Tensor, Mu: torch.Tensor, du: Optional[torch.Tensor] = None):
        self.graph, self.x, self.Mu, self.du = graph, x, Mu, du


class GRAND_plusConv(nn.Module):
    def __init__(self, opt, in_channels, out_channels, heads: int = 1, concat: bool = True, beta: bool = False,
                 dropout: float = 0.0, edge_dim: Optional[int] = None, bias: bool = True, root_weight: bool = True,
                 **kwargs):
        # **kwargs: the reference leaks `global_feat_dim=` into MessagePassing.__init__ (src/GNN.py:118)
        super().__init__()
        if heads != 1:
            raise NotImplementedError("heads > 1 is off the deformer hot path")
        if dropout != 0.0:
            raise NotImplementedError("attention dropout > 0 is off the deformer hot path")
        if edge_dim is not None:
            raise NotImplementedError("edge features are off the deformer hot path")
        if root_weight or beta:
            raise NotImplementedError("root_weight / beta are off the deformer hot path (GNN.py:118-119 sets them False)")
        if isinstance(in_channels, (tuple, list)):
            if in_channels[0] != in_channels[1]:
                raise NotImplementedError("bipartite in_channels are off the deformer hot path")
            in_channels = in_channels[0]
        if in_channels != out_channels:
            raise NotImplementedError("value = identity needs in_channels == out_channels (src/GRAND_plus.py:150)")
        if opt.get("reg_skew") and len(opt["mesh_dims"]) == 2:
            raise NotImplementedError("reg_skew needs the Firedrake mesh (src/GRAND_plus.py:280-324); not implemented")
        self.opt = opt
        self.dim = len(opt["mesh_dims"])
        self.in_channels, self.out_channels, self.heads = in_channels, out_channels, heads
        self.concat, self.beta, self.root_weight, self.dropout, self.edge_dim = concat, False, root_weight, dropout, edge_dim
        self.inv_temp = inv_temperature(opt)
        self.lin_key = nn.Linear(in_channels, heads * out_channels)
        self.lin_query = nn.Linear(in_channels, heads * out_channels)
        self.lin_value = nn.Identity()
        self.lin_skip = nn.Linear(in_channels, out_channels if not concat else heads * out_channels, bias=bias)
        if opt.get("softmax_temp_type") == "learnable_a":
            # `nn.Parameter(torch.Tensor(1, heads, 1))` in the reference (:154): uninitialised memory until a value is
            # loaded.  Same name and shape (a reference state_dict loads), initialised to opt['softmax_temp'].
            self.sm_temp_a = nn.Parameter(torch.full((1, heads, 1), float(opt.get("softmax_temp", 1.0))))
        self.reset_parameters()
        self.stored_ei = None
        self._alpha_src: Optional[_AlphaSource] = None
        self._alpha_cache = None
        self._graphs = GraphCache(capacity=4)

    def reset_parameters(self):
        self.lin_key.reset_parameters()
        self.lin_query.reset_parameters()
        self.lin_skip.reset_parameters()

    # ---- attention read-out -------------------------------------------------------------
    def _set_alpha_source(self, graph: MeshGraph, x: torch.Tensor, Mu: torch.Tensor, du: Optional[torch.Tensor] = None):
        self.stored_ei = graph.edge_index
        self._alpha_src = _AlphaSource(graph, x, Mu, du)
        self._alpha_cache = None

    @property
    def stored_alpha(self):
        """Attention weights [E, 1] of the last call, in `stored_ei` order (`src/GRAND_plus.py:253-256`)."""
        if self._alpha_cache is None and self._alpha_src is not None:
            s = self._alpha_src
            self._alpha_cache = GF.conv_alpha(s.graph, s.x, s.Mu, s.du).view(-1, 1)
        return self._alpha_cache

    @stored_alpha.setter
    def stored_alpha(self, value):
        self._alpha_cache = value
        self._alpha_src = None

    # ---- operator ------------------------------------------------------------------------
    def _graph_for(self, edge_index: torch.Tensor, num_nodes: int) -> MeshGraph:
        key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version, num_nodes, str(edge_index.device))
        g = self._graphs.get(key)
        if g is None:
            g = MeshGraph.build(edge_index, num_nodes)
            self._graphs.put(key, g, (edge_index,))
        return g

    def forward(self, x, edge_index, global_features=None, mesh=None, edge_attr=None, return_attention_weights=None):
        if isinstance(x, (tuple, list)):
            x = x[0]
        if edge_attr is not None:
            raise NotImplementedError("edge_attr is off the deformer hot path")
        if x.device.type != "cuda":
            raise RuntimeError("GRAND_plusConv runs on CUDA only: the sm_100a kernels have no CPU fallback")
        if self.opt.get("softmax_temp_type") == "learnable_a":
            raise NotImplementedError("softmax_temp_type='learnable_a' is implemented on the module seam (GNN.forward); "
                                      "the single-layer operator seam takes a fixed temperature")
        graph = edge_index if isinstance(edge_index, MeshGraph) else self._graph_for(edge_index, x.shape[0])
        res = GF.ConvFunction.apply(x, self.lin_query.weight, self.lin_query.bias, self.lin_key.weight,
                                    self.lin_key.bias, graph, self.inv_temp)
        if isinstance(self.opt.get("show_mesh_evol_plots"), bool) or isinstance(return_attention_weights, bool):
            _, CE = GF.live_channels(x.shape[1], x.shape[1])
            xp = x.detach()
            if CE != x.shape[1]:
                xp = torch.nn.functional.pad(xp, (0, CE - x.shape[1]))
            Mu = GF.prepare_weights(self.lin_query.weight.detach().unsqueeze(0), self.lin_query.bias.detach().unsqueeze(0),
                                    self.lin_key.weight.detach().unsqueeze(0), CE, self.inv_temp)
            self._set_alpha_source(graph, xp.float().contiguous(), Mu)
        if isinstance(return_attention_weights, bool):
            return res, (graph.edge_index, self.stored_alpha)
        return res

    def __repr__(self) -> str:
        return f"{self.__class__.__name__}({self.in_channels}, {self.out_channels}, heads={self.heads})"


class GRAND_conv(GRAND_plusConv):
    """`GRAND_conv` (`src/GRAND_plus.py:366-382`): TransformerConv with identity value -- the same
    arithmetic without temperature / reg_skew; `forward(x, edge_index)` returns `A x - x`."""

    def __init__(self, opt, in_channels, out_channels, heads=1, concat=False, beta=False, dropout=0,
                 edge_dim=None, bias=False, root_weight=False):
        plain = dict(opt)
        plain["softmax_temp_type"] = None
        plain["reg_skew"] = False
        plain["show_mesh_evol_plots"] = True   # return_attention_weights=True stores ei / alpha every call (:381)
        super().__init__(plain, in_channels, out_channels, heads=1, concat=False, beta=False, dropout=0.0,
                         edge_dim=None, bias=False, root_weight=False)
        self.opt = opt

    def forward(self, x, edge_index):
        opt, self.opt = self.opt, {"show_mesh_evol_plots": True}
        try:
            return super().forward(x, edge_index)
        finally:
            self.opt = opt
