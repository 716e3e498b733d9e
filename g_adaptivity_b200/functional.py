"""Thin Python wrappers over the C-ABI calls + the autograd glue.

Everything here is plumbing: tensors are allocated with torch, their device pointers and the
current CUDA stream are handed to `libgadapt_b200.so`.  No arithmetic of the hot path is done in
PyTorch.  All functions require CUDA tensors and raise otherwise.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch

from . import _lib
from .graph import MeshGraph

METHOD_EULER, METHOD_RK4 = 0, 1
METHODS = {"euler": METHOD_EULER, "rk4": METHOD_RK4}


def live_channels(in_dim: int, hidden_dim: int) -> Tuple[int, int]:
    """(number of live channels, padded vector width CE).  With the identity encoder
    (`src/GNN.py:75-90`) only the first min(in_dim, hidden_dim) channels are ever non-zero."""
    live = min(int(in_dim), int(hidden_dim))
    for ce in (2, 4, 8):
        if live <= ce:
            return live, ce
    raise NotImplementedError(f"{live} live channels: the sm_100a kernels are instantiated for <= 8")


def use_ell(graph: MeshGraph, CE: int) -> bool:
    """True when the mesh-resident ELL kernels serve this graph (bounded degree, tiles planned,
    ELL rows built for this channel width); otherwise the CSR mesh-resident / streaming kernels do."""
    return graph.ell_in is not None and graph.ell_ce == CE and graph.tile_ptr is not None


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream(t: torch.Tensor) -> int:
    """cudaStream_t of the tensor's device's current stream (the raw getter skips building a Stream object: this is on
    the host path of every module call)."""
    if _raw_stream is not None:
        return _raw_stream(t.device.index if t.device.index is not None else torch.cuda.current_device())
    return torch.cuda.current_stream(t.device).cuda_stream


class _NoSwitch:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NO_SWITCH = _NoSwitch()


def _on_device(dev):
    """`torch.cuda.device(dev)` only when `dev` is not the current device already (the context manager costs several
    microseconds of host time on every call otherwise)."""
    idx = dev.index if isinstance(dev, torch.device) else dev
    if idx is None or idx == torch.cuda.current_device():
        return _NO_SWITCH
    return torch.cuda.device(idx)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and t.device.type != "cuda":
            raise RuntimeError("g_adaptivity_b200 kernels need CUDA tensors (there is no CPU fallback)")


def _f32(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ------------------------------------------------------------------------------------------
def prepare_weights(Wq: torch.Tensor, bq: torch.Tensor, Wk: torch.Tensor, CE: int, inv_temp: float) -> torch.Tensor:
    """[Lw, C, C], [Lw, C], [Lw, C, C] -> Mu [Lw, CE*CE + CE]  (see csrc/weights.cu)."""
    _need_cuda(Wq, bq, Wk)
    lib = _lib.load()
    Wq, bq, Wk = _f32(Wq), _f32(bq), _f32(Wk)
    Lw, C = Wq.shape[0], Wq.shape[1]
    Mu = torch.empty((Lw, CE * CE + CE), dtype=torch.float32, device=Wq.device)
    with _on_device(Wq.device):
        _lib.check(lib.gad_prepare_weights(_lib.ptr(Wq), _lib.ptr(bq), _lib.ptr(Wk), Lw, C, CE, float(inv_temp),
                                           _lib.ptr(Mu), _stream(Wq)), "gad_prepare_weights")
    return Mu


def weight_grads(Wq, bq, Wk, gMu, CE: int, inv_temp: float):
    lib = _lib.load()
    Wq, bq, Wk = _f32(Wq), _f32(bq), _f32(Wk)
    Lw, C = Wq.shape[0], Wq.shape[1]
    gWq, gWk = torch.empty_like(Wq), torch.empty_like(Wk)
    gbq, gbk = torch.empty_like(bq), torch.empty_like(bq)
    with _on_device(Wq.device):
        _lib.check(lib.gad_weight_grads(_lib.ptr(Wq), _lib.ptr(bq), _lib.ptr(Wk), _lib.ptr(gMu), Lw, C, CE,
                                        float(inv_temp), _lib.ptr(gWq), _lib.ptr(gbq), _lib.ptr(gWk), _lib.ptr(gbk),
                                        _stream(Wq)), "gad_weight_grads")
    return gWq, gbq, gWk, gbk


def pack_features(x_comp, f, uu, f_scale, uu_scale, CE: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`features = cat[x_comp, f, uu]` + identity encoder (`src/GNN.py:225-239,270`) -> x0 [N, CE]."""
    _need_cuda(x_comp, f, uu)
    lib = _lib.load()
    x_comp = _f32(x_comp)
    if x_comp.dim() == 1:
        x_comp = x_comp.unsqueeze(-1)
    N, dim = x_comp.shape
    f, uu = _f32(f), _f32(uu)
    if out is None:
        out = torch.empty((N, CE), dtype=torch.float32, device=x_comp.device)
    with _on_device(x_comp.device):
        _lib.check(lib.gad_pack_features(_lib.ptr(x_comp), _lib.ptr(f), _lib.ptr(uu), _lib.ptr(f_scale),
                                         _lib.ptr(uu_scale), N, dim, CE, _lib.ptr(out), _stream(x_comp)),
                   "gad_pack_features")
    return out


def deform_forward(graph: MeshGraph, x0: torch.Tensor, dim: int, Mu: torch.Tensor, tau: torch.Tensor,
                   method: int = METHOD_EULER, states: Optional[torch.Tensor] = None,
                   force_stream: bool = False, du: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x0 [N, CE] -> x_phys [N, dim].  `states` ([L, N, CE], states[0] aliasing x0) receives the
    layer inputs x^0..x^{L-1} for the backward.  `du` [meshes, Lw, CE]: per-mesh bias offset (see _check_du)."""
    _need_cuda(x0, Mu, tau)
    lib = _lib.load()
    N, CE = x0.shape
    L, Lw = int(tau.numel()), int(Mu.shape[0])
    assert graph.N == N
    x_phys = torch.empty((N, dim), dtype=torch.float32, device=x0.device)
    use_tiles = graph.tile_ptr is not None and not force_stream
    if du is not None:
        _check_du(graph, du, CE, Lw, force_stream)
        if use_tiles:
            raise NotImplementedError("deform_forward takes the bias offset on the streaming kernels only; "
                                      "use deform_forward_raw on mesh-resident graphs")
    if use_tiles and use_ell(graph, CE):
        with _on_device(x0.device):
            _lib.check(lib.gad_deform_fwd_ell(
                _lib.ptr(graph.ell_in), N, _lib.ptr(graph.ell_tile_ptr), graph.T, graph.max_tile_nodes, graph.ell_deg,
                _lib.ptr(x0), dim, CE, _lib.ptr(Mu), Lw, _lib.ptr(tau), L, method, _lib.ptr(x_phys),
                _lib.ptr(states), _stream(x0)), "gad_deform_fwd_ell")
        return x_phys
    ws = None
    ws_bytes = 0
    if not use_tiles:
        _need_wide(graph, CE, du)
        ws_bytes = lib.gad_deform_workspace_bytes(N, CE, method)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x0.device)
        if graph.ensure_wide(CE):      # streaming ELL kernels (csrc/stream_ell.cu)
            with _on_device(x0.device):
                _lib.check(lib.gad_deform_fwd_wide(
                    _lib.ptr(graph.wide_in), N, graph.wide_deg, graph.wide_reach, _lib.ptr(x0), dim, CE, _lib.ptr(Mu),
                    _lib.ptr(du), _n_meshes(graph, du), Lw, _lib.ptr(tau), L, method, _lib.ptr(x_phys), _lib.ptr(states),
                    _lib.ptr(ws), ws_bytes, _stream(x0)), "gad_deform_fwd_wide")
            return x_phys
    with _on_device(x0.device):
        _lib.check(lib.gad_deform_fwd(
            _lib.ptr(graph.rowptr), _lib.ptr(graph.col_walk), N, graph.E,
            _lib.ptr(graph.tile_ptr) if use_tiles else None, graph.T if use_tiles else 0,
            graph.max_tile_nodes, graph.max_tile_edges, _lib.ptr(x0), dim, CE, _lib.ptr(Mu), Lw, _lib.ptr(tau), L,
            method, _lib.ptr(x_phys), _lib.ptr(states), _lib.ptr(ws), ws_bytes, _stream(x0)), "gad_deform_fwd")
    return x_phys


def fold_scale(inv_temp: float, C: int) -> float:
    """Scale of the folded logits (csrc/tail_math.cuh: fold_scale): log2(e) * inv_temp / sqrt(C)."""
    import math
    return math.log2(math.e) * float(inv_temp) / math.sqrt(float(C))


def _check_du(graph: MeshGraph, du: torch.Tensor, CE: int, Lw: int, force_stream: bool):
    """Per-mesh bias offsets du [meshes, Lw, CE] (global CNN features, include/gadapt.h) run on the mesh-resident ELL
    kernels with one mesh per tile, on the cluster kernels and on the streaming ELL kernels (meshes of one size); the
    CSR kernels take none."""
    if graph.mesh_sizes is None:
        raise NotImplementedError("global CNN features need the batch's mesh sizes")
    M = len(graph.mesh_sizes)
    if graph.tile_ptr is not None and not force_stream:
        if not use_ell(graph, CE):
            raise NotImplementedError("global CNN features (per-mesh bias offset) do not run on the CSR mesh-resident "
                                      "kernels (degree > 7 or CE = 8)")
        if graph.T != M:
            raise NotImplementedError("global CNN features need one mesh per tile (the module plans tiles that way)")
    elif any(n != graph.mesh_sizes[0] for n in graph.mesh_sizes) or CE not in (2, 4) or max(graph.max_in_deg, graph.max_out_deg) > 7:
        raise NotImplementedError("global CNN features on meshes beyond one CTA need meshes of equal size, degree <= 7 and "
                                  "CE in {2, 4} (the CSR streaming kernels take no bias offset)")
    if tuple(du.shape) != (M, Lw, CE) or du.dtype != torch.float32 or not du.is_contiguous():
        raise ValueError(f"du must be a contiguous float32 [{M}, {Lw}, {CE}] tensor, got {tuple(du.shape)}")


def _n_meshes(graph: MeshGraph, du: Optional[torch.Tensor]) -> int:
    """The mesh count the streaming entry points take with `du` (0 without)."""
    return len(graph.mesh_sizes) if du is not None else 0


def _need_wide(graph: MeshGraph, CE: int, du: Optional[torch.Tensor]):
    """With `du`, the streaming route must be the wide-row one: the CSR streaming kernels take no offset."""
    if du is not None and not graph.ensure_wide(CE):
        raise NotImplementedError("global CNN features (per-mesh bias offset) need the streaming ELL kernels "
                                  "(degree <= 7, CE in {2, 4}); the CSR streaming kernels take none")


def deform_forward_raw(graph: MeshGraph, x_comp, f, uu, f_scale, uu_scale, dim: int, CE: int, Mu: torch.Tensor,
                       tau: torch.Tensor, method: int = METHOD_EULER, states: Optional[torch.Tensor] = None,
                       force_stream: bool = False, du: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw inputs -> x_phys [N, dim]: on mesh-resident ELL graphs ONE launch (feature assembly fused
    into the forward kernel's input staging, csrc/ell_kernels.cuh); otherwise pack + forward."""
    _need_cuda(x_comp, f, uu, Mu, tau)
    x_comp = _f32(x_comp)
    if x_comp.dim() == 1:
        x_comp = x_comp.unsqueeze(-1)
    N = x_comp.shape[0]
    if du is not None:
        _check_du(graph, du, CE, int(Mu.shape[0]), force_stream)
    if (graph.tile_ptr is None and not force_stream and not getattr(graph, "_no_cluster", False)
            and graph.ensure_cluster_fwd(CE)
            and not graph.stream_fwd_preferred(CE, int(tau.numel()) * (4 if method == METHOD_RK4 else 1))):
        # meshes beyond one CTA: one thread-block cluster per mesh, ONE launch for all layers / RK4 steps
        lib = _lib.load()
        if f is not None and dim >= CE:
            f = None
        if uu is not None and dim + (1 if f is not None else 0) >= CE:
            uu = None
        f, uu = _f32(f), _f32(uu)
        L, Lw = int(tau.numel()), int(Mu.shape[0])
        x_phys = torch.empty((N, dim), dtype=torch.float32, device=x_comp.device)
        with _on_device(x_comp.device):
            _lib.check(lib.gad_deform_fwd_cluster(
                _lib.ptr(graph.clf_in), _lib.ptr(graph.clf_mesh_ptr), len(graph.mesh_sizes), max(graph.mesh_sizes),
                graph.clf_deg, graph.clf_C, N, _lib.ptr(x_comp), _lib.ptr(f), _lib.ptr(uu), _lib.ptr(f_scale),
                _lib.ptr(uu_scale), dim, CE, _lib.ptr(Mu), _lib.ptr(du), Lw, _lib.ptr(tau), L, method, _lib.ptr(x_phys),
                _lib.ptr(states), _stream(x_comp)), "gad_deform_fwd_cluster")
        return x_phys
    if not (graph.tile_ptr is not None and not force_stream and use_ell(graph, CE)):
        x0 = states[0] if states is not None else torch.empty((N, CE), dtype=torch.float32, device=x_comp.device)
        pack_features(x_comp, f, uu, f_scale, uu_scale, CE, out=x0)
        return deform_forward(graph, x0, dim, Mu, tau, method, states=states, force_stream=force_stream, du=du)
    lib = _lib.load()
    # identity encoder with hidden < in_dim truncates (src/GNN.py:84-90): features beyond CE are dropped
    if f is not None and dim >= CE:
        f = None
    if uu is not None and dim + (1 if f is not None else 0) >= CE:
        uu = None
    f, uu = _f32(f), _f32(uu)
    L, Lw = int(tau.numel()), int(Mu.shape[0])
    assert graph.N == N
    x_phys = torch.empty((N, dim), dtype=torch.float32, device=x_comp.device)
    with _on_device(x_comp.device):
        _lib.check(lib.gad_deform_fwd_ell_raw(
            _lib.ptr(graph.ell_in), N, _lib.ptr(graph.ell_tile_ptr), graph.T, graph.max_tile_nodes, graph.ell_deg,
            _lib.ptr(x_comp), _lib.ptr(f), _lib.ptr(uu), _lib.ptr(f_scale), _lib.ptr(uu_scale), dim, CE, _lib.ptr(Mu),
            _lib.ptr(du), Lw, _lib.ptr(tau), L, method, _lib.ptr(x_phys), _lib.ptr(states), _stream(x_comp)),
            "gad_deform_fwd_ell_raw")
    return x_phys


def _tile_bias_grads(ws: torch.Tensor, T: int, Lw: int, L: int, CE: int) -> torch.Tensor:
    """d loss / d du [T, Lw, CE] from the backward's workspace: it begins with the per-tile partials
    [T, slots, CE*CE + CE + 1] (include/gadapt.h), whose entries CE*CE .. CE*CE + CE - 1 are sum_i t_i of the tile."""
    slots, nacc = (L if Lw > 1 else 1), CE * CE + CE + 1
    part = ws[:T * slots * nacc * 4].view(torch.float32).view(T, slots, nacc)
    return part[:, :, CE * CE:CE * CE + CE].clone()


def rk4_backward_resident(graph: MeshGraph, CE: int, force_stream: bool = False) -> bool:
    """Which kernel runs the backward through RK4 steps on `graph`: True for the mesh-resident one
    (csrc/ell_kernels.cuh: k_ell_bwd_rk4, gad_deform_bwd_ell_rk4), False for the streaming chain
    (csrc/stream_ell.cu, gad_deform_bwd_wide_rk4; its wide rows are built here, so call this outside any capture).
    Raises NotImplementedError when neither serves the graph.  The module path and DeformerTrainer both ask here."""
    lib = _lib.load()
    if (graph.tile_ptr is not None and not force_stream and use_ell(graph, CE)
            and lib.gad_ell_rk4_bwd_supported(CE, graph.max_tile_nodes, graph.ell_deg)):
        return True
    if not graph.ensure_wide(CE):
        raise NotImplementedError(
            "backward through ode_method='rk4': meshes of at most ~1200 nodes run on the mesh-resident ELL kernel, "
            "larger ones on the streaming ELL kernels, both for degree <= 7 and 2 or 4 live channels; this graph "
            f"has max degree {max(graph.max_in_deg, graph.max_out_deg)}, CE = {CE}")
    return False


def deform_backward_rk4(graph: MeshGraph, states: torch.Tensor, g_xphys: torch.Tensor, dim: int, Mu: torch.Tensor,
                        tau: torch.Tensor, want_gx0: bool = False, du: Optional[torch.Tensor] = None,
                        force_stream: bool = False):
    """Backward through classical RK4 steps: cotangent of x_phys -> (gMu, g_x0 | None, g_du | None).  Meshes that fit a
    CTA: one launch of the mesh-resident kernel (csrc/ell_kernels.cuh: k_ell_bwd_rk4).  Larger meshes (or
    `force_stream`): the streaming kernels, three stage recomputes and four vjp passes per step
    (csrc/stream_ell.cu: wide_backward_rk4_t).  The step sizes get no gradient (learn_step is an Euler feature)."""
    _need_cuda(states, g_xphys, Mu, tau)
    lib = _lib.load()
    L, N, CE = states.shape
    Lw = int(Mu.shape[0])
    g_xphys = _f32(g_xphys)
    dev = states.device
    gMu = torch.empty_like(Mu)
    g_x0 = torch.empty((N, CE), dtype=torch.float32, device=dev) if want_gx0 else None
    if not rk4_backward_resident(graph, CE, force_stream):
        ws_bytes = lib.gad_deform_bwd_wide_rk4_workspace_bytes(N, CE)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        g_du = torch.empty_like(du) if du is not None else None
        with _on_device(dev):
            _lib.check(lib.gad_deform_bwd_wide_rk4(
                _lib.ptr(graph.wide_in), _lib.ptr(graph.wide_out), N, graph.wide_deg, _lib.ptr(states), _lib.ptr(g_xphys),
                dim, CE, _lib.ptr(Mu), _lib.ptr(du), _n_meshes(graph, du), Lw, _lib.ptr(tau), L, _lib.ptr(gMu),
                _lib.ptr(g_x0), _lib.ptr(g_du), _lib.ptr(ws), ws_bytes, _stream(states)), "gad_deform_bwd_wide_rk4")
        return gMu, g_x0, g_du
    ws_bytes = lib.gad_ell_workspace_bytes(CE, graph.T, L)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with _on_device(dev):
        _lib.check(lib.gad_deform_bwd_ell_rk4(
            _lib.ptr(graph.ell_in), _lib.ptr(graph.ell_out), N, _lib.ptr(graph.ell_tile_ptr), graph.T,
            graph.max_tile_nodes, graph.ell_deg, _lib.ptr(states), _lib.ptr(g_xphys), dim, CE, _lib.ptr(Mu), _lib.ptr(du),
            Lw, _lib.ptr(tau), L, _lib.ptr(gMu), _lib.ptr(g_x0), _lib.ptr(ws), ws_bytes, _stream(states)),
            "gad_deform_bwd_ell_rk4")
    g_du = _tile_bias_grads(ws, graph.T, Lw, L, CE) if du is not None else None
    return gMu, g_x0, g_du


def deform_backward(graph: MeshGraph, states: torch.Tensor, g_xphys: torch.Tensor, dim: int, Mu: torch.Tensor,
                    tau: torch.Tensor, want_gtau: bool = False, want_gx0: bool = False, force_stream: bool = False,
                    du: Optional[torch.Tensor] = None):
    """Cotangent of x_phys -> (gMu [Lw, CE*CE+CE], g_tau [L] | None, g_x0 [N, CE] | None[, g_du [meshes, Lw, CE]])."""
    _need_cuda(states, g_xphys, Mu, tau)
    lib = _lib.load()
    L, N, CE = states.shape
    Lw = int(Mu.shape[0])
    g_xphys = _f32(g_xphys)
    dev = states.device
    gMu = torch.empty_like(Mu)
    g_tau = torch.empty(L, dtype=torch.float32, device=dev) if want_gtau else None
    g_x0 = torch.empty((N, CE), dtype=torch.float32, device=dev) if want_gx0 else None
    use_tiles = graph.tile_ptr is not None and not force_stream
    T = graph.T if use_tiles else 0
    if use_tiles and use_ell(graph, CE):
        ws_bytes = lib.gad_ell_workspace_bytes(CE, T, L)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with _on_device(dev):
            _lib.check(lib.gad_deform_bwd_ell(
                _lib.ptr(graph.ell_in), _lib.ptr(graph.ell_out), N, _lib.ptr(graph.ell_tile_ptr), T,
                graph.max_tile_nodes, graph.ell_deg, _lib.ptr(states), _lib.ptr(g_xphys), dim, CE, _lib.ptr(Mu),
                _lib.ptr(du), Lw, _lib.ptr(tau), L, _lib.ptr(gMu), _lib.ptr(g_tau), _lib.ptr(g_x0), _lib.ptr(ws), ws_bytes,
                _stream(states)), "gad_deform_bwd_ell")
        if du is not None:
            return gMu, g_tau, g_x0, _tile_bias_grads(ws, T, Lw, L, CE)
        return gMu, g_tau, g_x0
    g_du = torch.empty_like(du) if du is not None else None
    done = (gMu, g_tau, g_x0) if du is None else (gMu, g_tau, g_x0, g_du)
    if (graph.tile_ptr is None and not force_stream and not getattr(graph, "_no_cluster", False)
            and graph.ensure_cluster(CE)):
        # meshes beyond one CTA (up to 4 slabs): cluster-resident backward, one launch + the reduction
        M = len(graph.mesh_sizes)
        ws_bytes = lib.gad_cluster_workspace_bytes(CE, M, graph.cl_C, L)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with _on_device(dev):
            _lib.check(lib.gad_deform_bwd_cluster(
                _lib.ptr(graph.cl_in), _lib.ptr(graph.cl_out), _lib.ptr(graph.mesh_ptr), M, max(graph.mesh_sizes),
                graph.cl_deg, graph.cl_C, N, _lib.ptr(states), _lib.ptr(g_xphys), dim, CE, _lib.ptr(Mu), _lib.ptr(du), Lw,
                _lib.ptr(tau), L, _lib.ptr(gMu), _lib.ptr(g_tau), _lib.ptr(g_x0), _lib.ptr(g_du), _lib.ptr(ws), ws_bytes,
                _stream(states)), "gad_deform_bwd_cluster")
        return done
    ws_bytes = lib.gad_deform_bwd_workspace_bytes(N, CE, T, L)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    if not use_tiles:
        _need_wide(graph, CE, du)
    if not use_tiles and graph.ensure_wide(CE):
        with _on_device(dev):
            _lib.check(lib.gad_deform_bwd_wide(
                _lib.ptr(graph.wide_in), _lib.ptr(graph.wide_out), N, graph.wide_deg, _lib.ptr(states), _lib.ptr(g_xphys),
                dim, CE, _lib.ptr(Mu), _lib.ptr(du), _n_meshes(graph, du), Lw, _lib.ptr(tau), L, _lib.ptr(gMu),
                _lib.ptr(g_tau), _lib.ptr(g_x0), _lib.ptr(g_du), _lib.ptr(ws), ws_bytes, _stream(states)),
                "gad_deform_bwd_wide")
        return done
    if du is not None:
        raise NotImplementedError("global CNN features (per-mesh bias offset) do not run on the CSR kernels")
    with _on_device(dev):
        _lib.check(lib.gad_deform_bwd(
            _lib.ptr(graph.rowptr), _lib.ptr(graph.col_walk), _lib.ptr(graph.t_rowptr), _lib.ptr(graph.t_dst_walk), N, graph.E,
            _lib.ptr(graph.tile_ptr) if use_tiles else None, T, graph.max_tile_nodes, graph.max_tile_edges,
            _lib.ptr(states), _lib.ptr(g_xphys), dim, CE, _lib.ptr(Mu), Lw, _lib.ptr(tau), L, _lib.ptr(gMu),
            _lib.ptr(g_tau), _lib.ptr(g_x0), _lib.ptr(ws), ws_bytes, _stream(states)), "gad_deform_bwd")
    return gMu, g_tau, g_x0


def conv_forward(graph: MeshGraph, x: torch.Tensor, Mu: torch.Tensor, want_res: bool = True,
                 want_alpha: bool = False):
    """One layer: res = A(x) x - x  [N, CE];  alpha [E] in filtered edge-list order."""
    _need_cuda(x, Mu)
    lib = _lib.load()
    N, CE = x.shape
    res = torch.empty_like(x) if want_res else None
    alpha = torch.empty(graph.E, dtype=torch.float32, device=x.device) if want_alpha else None
    with _on_device(x.device):
        _lib.check(lib.gad_conv_fwd(_lib.ptr(graph.rowptr), _lib.ptr(graph.col), _lib.ptr(graph.eid), N, graph.E,
                                    _lib.ptr(x), CE, _lib.ptr(Mu), _lib.ptr(res), _lib.ptr(alpha), _stream(x)),
                   "gad_conv_fwd")
    return res, alpha


def conv_alpha(graph: MeshGraph, x: torch.Tensor, Mu: torch.Tensor, du: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Attention weights alpha [E] of one layer in filtered edge-list order.  `du` [meshes, CE] (or None): the per-mesh
    bias offset of this layer's weight set that the deformer ran with (global CNN features, meshes of equal size)."""
    if du is None:
        return conv_forward(graph, x, Mu, want_res=False, want_alpha=True)[1]
    _need_cuda(x, Mu, du)
    lib = _lib.load()
    N, CE = x.shape
    du = _f32(du)
    if graph.mesh_sizes is None or du.shape != (len(graph.mesh_sizes), CE):
        raise ValueError(f"du must be [meshes, {CE}], got {tuple(du.shape)}")
    alpha = torch.empty(graph.E, dtype=torch.float32, device=x.device)
    with _on_device(x.device):
        _lib.check(lib.gad_conv_alpha_du(_lib.ptr(graph.rowptr), _lib.ptr(graph.col), _lib.ptr(graph.eid), N, graph.E,
                                         _lib.ptr(x), CE, _lib.ptr(Mu), _lib.ptr(du), int(du.shape[0]), _lib.ptr(alpha),
                                         _stream(x)), "gad_conv_alpha_du")
    return alpha


def conv_backward(graph: MeshGraph, x: torch.Tensor, g_res: torch.Tensor, Mu: torch.Tensor):
    lib = _lib.load()
    N, CE = x.shape
    gMu = torch.empty_like(Mu)
    g_x = torch.empty_like(x)
    ws_bytes = lib.gad_deform_bwd_workspace_bytes(N, CE, 0, 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
    with _on_device(x.device):
        _lib.check(lib.gad_conv_bwd(_lib.ptr(graph.rowptr), _lib.ptr(graph.col), _lib.ptr(graph.t_rowptr),
                                    _lib.ptr(graph.t_dst), N, graph.E, _lib.ptr(x), _lib.ptr(_f32(g_res)), CE,
                                    _lib.ptr(Mu), _lib.ptr(gMu), _lib.ptr(g_x), _lib.ptr(ws), ws_bytes, _stream(x)),
                   "gad_conv_bwd")
    return gMu, g_x


def mesh_loss(out: torch.Tensor, target: torch.Tensor, kind: str = "l1", want_grad: bool = True):
    """mean |out - target| (or squared), plus d loss / d out -- `run_GNN.py:80-84,103-106`."""
    _need_cuda(out, target)
    lib = _lib.load()
    out, target = _f32(out), _f32(target)
    if target.dim() == 1:
        target = target.unsqueeze(-1)
    assert out.shape == target.shape
    count = out.numel()
    loss = torch.empty(1, dtype=torch.float32, device=out.device)
    g = torch.empty_like(out) if want_grad else None
    ws = torch.empty(lib.gad_mesh_loss_workspace_bytes(count), dtype=torch.uint8, device=out.device)
    with _on_device(out.device):
        _lib.check(lib.gad_mesh_loss(_lib.ptr(out), _lib.ptr(target), count, 0 if kind == "l1" else 1,
                                     1.0 / count, _lib.ptr(loss), _lib.ptr(g), _lib.ptr(ws), _stream(out)),
                   "gad_mesh_loss")
    return loss, g


# ------------------------------------------------------------------------------------------
# autograd glue
# ------------------------------------------------------------------------------------------
class DeformFunction(torch.autograd.Function):
    """x_phys = Deformer(x_comp, f, uu; Wq, bq, Wk, bk, tau) with hand-written backward kernels.

    Differentiable inputs: Wq, bq, Wk, bk (gradient identically zero), tau, and -- when they
    require grad and no normalisation is active -- x_comp / f / uu."""

    @staticmethod
    def forward(ctx, x_comp, f, uu, f_scale, uu_scale, Wq, bq, Wk, bk, tau, graph, dim, CE, inv_temp, method,
                force_stream, aux, du=None, temp=None):
        L = int(tau.numel())
        N = x_comp.shape[0]
        needs = any(ctx.needs_input_grad)
        tau_d = _f32(tau.detach().reshape(-1))
        Mu = aux.get("Mu_in") if aux is not None else None     # folded weights cached by the module
        if Mu is None:
            Mu = prepare_weights(Wq.detach(), bq.detach(), Wk.detach(), CE, inv_temp)
        # learnable temperature (softmax_temp_type='learnable_a'): the logits are divided by T_l, i.e. the folded
        # weights of set l are scaled by 1 / T_l -- (M, u) are linear in the logit scale
        ctx.has_temp = temp is not None
        if temp is not None:
            inv_t = (1.0 / temp.detach().float().reshape(-1, 1))
            Mu = (Mu * inv_t).contiguous()
        keep_states = aux is not None and aux.get('keep_states', False)
        states = torch.empty((L, N, CE), dtype=torch.float32, device=x_comp.device) if (needs or keep_states) else None
        x_phys = deform_forward_raw(graph, x_comp.detach(), None if f is None else f.detach(),
                                    None if uu is None else uu.detach(), f_scale, uu_scale, dim, CE, Mu, tau_d, method,
                                    states=states, force_stream=force_stream,
                                    du=None if du is None else du.detach().float().contiguous())
        ctx.method = method
        ctx.has_du = du is not None
        ctx.graph, ctx.dim, ctx.CE, ctx.inv_temp, ctx.force_stream = graph, dim, CE, inv_temp, force_stream
        ctx.has_f, ctx.has_uu = f is not None, uu is not None
        ctx.normalised = (f_scale is not None) or (uu_scale is not None)
        if needs:
            ctx.save_for_backward(states, Mu, tau_d, Wq, bq, Wk,
                                  du.detach().float().contiguous() if du is not None else torch.empty(0, device=Mu.device),
                                  temp.detach().float().reshape(-1) if temp is not None else torch.empty(0, device=Mu.device))
        if aux is not None:   # side channel for the lazy attention read-out (conv.stored_alpha)
            aux["states"], aux["Mu"] = (states if keep_states else None), Mu
        return x_phys

    @staticmethod
    def backward(ctx, g_xphys):
        states, Mu, tau_d, Wq, bq, Wk = ctx.saved_tensors[:6]
        du = ctx.saved_tensors[6] if ctx.has_du else None
        temp = ctx.saved_tensors[7] if ctx.has_temp else None
        g_du = g_temp = None
        ni = ctx.needs_input_grad
        want_gx0 = ni[0] or ni[1] or ni[2]
        if want_gx0 and ctx.normalised:
            raise NotImplementedError("input gradients with gnn_normalize=True are not implemented")
        if ctx.method == METHOD_RK4:
            if ni[9]:
                raise NotImplementedError("learn_step with ode_method='rk4': the step sizes get no gradient through RK4")
            gMu, g_x0, g_du = deform_backward_rk4(ctx.graph, states, g_xphys.contiguous(), ctx.dim, Mu, tau_d,
                                                  want_gx0=want_gx0, du=du, force_stream=ctx.force_stream)
            g_tau = None
        else:
            res = deform_backward(ctx.graph, states, g_xphys.contiguous(), ctx.dim, Mu, tau_d,
                                  want_gtau=ni[9], want_gx0=want_gx0, force_stream=ctx.force_stream, du=du)
            gMu, g_tau, g_x0 = res[:3]
            g_du = res[3] if du is not None else None
        if temp is not None:
            # Mu_l = Mu_base_l / T_l:  dL/dT_l = -<gMu_l, Mu_l> / T_l ,  dL/dMu_base_l = gMu_l / T_l
            g_temp = (-(gMu * Mu).sum(dim=1) / temp).reshape(-1)
            gMu = (gMu / temp.reshape(-1, 1)).contiguous()
        gWq, gbq, gWk, gbk = weight_grads(Wq.detach(), bq.detach(), Wk.detach(), gMu, ctx.CE, ctx.inv_temp)
        g_xc = g_f = g_uu = None
        if want_gx0:
            c = ctx.dim
            if ni[0]:
                g_xc = g_x0[:, :ctx.dim]
            if ctx.has_f:
                if ni[1] and c < ctx.CE:
                    g_f = g_x0[:, c]
                c += 1
            if ctx.has_uu and ni[2] and c < ctx.CE:
                g_uu = g_x0[:, c]
        return (g_xc, g_f, g_uu, None, None, gWq if ni[5] else None, gbq if ni[6] else None,
                gWk if ni[7] else None, gbk if ni[8] else None,
                g_tau.view_as(tau_d) if (ni[9] and g_tau is not None) else None,
                None, None, None, None, None, None, None, g_du, g_temp)


class ConvFunction(torch.autograd.Function):
    """Operator seam: res = A(x) x - x for one GRAND_plusConv / GRAND_conv layer."""

    @staticmethod
    def forward(ctx, x, Wq, bq, Wk, bk, graph, inv_temp):
        N, C = x.shape
        _, CE = live_channels(C, C)
        xp = x.detach()
        if CE != C:
            xp = torch.nn.functional.pad(xp, (0, CE - C))
        xp = _f32(xp)
        Mu = prepare_weights(Wq.detach().unsqueeze(0), bq.detach().unsqueeze(0), Wk.detach().unsqueeze(0), CE, inv_temp)
        res, _ = conv_forward(graph, xp, Mu)
        ctx.graph, ctx.C, ctx.CE, ctx.inv_temp = graph, C, CE, inv_temp
        ctx.save_for_backward(xp, Mu, Wq, bq, Wk)
        return res[:, :C] if CE != C else res

    @staticmethod
    def backward(ctx, g_res):
        xp, Mu, Wq, bq, Wk = ctx.saved_tensors
        g = g_res.contiguous()
        if ctx.CE != ctx.C:
            g = torch.nn.functional.pad(g, (0, ctx.CE - ctx.C))
        gMu, g_x = conv_backward(ctx.graph, xp, g, Mu)
        gWq, gbq, gWk, gbk = weight_grads(Wq.detach().unsqueeze(0), bq.detach().unsqueeze(0),
                                          Wk.detach().unsqueeze(0), gMu, ctx.CE, ctx.inv_temp)
        return (g_x[:, :ctx.C] if ctx.CE != ctx.C else g_x, gWq[0], gbq[0], gWk[0], gbk[0], None, None)
