"""Data-parallel training step of the deformer, CUDA-graph captured.

The reference trains with the loop of `src/run_GNN.py:95-131` (forward, L1 mesh loss, autograd
backward, `torch.optim.Adam`), single process.  `DeformerTrainer` runs the same step as one
replayable CUDA graph per resident batch ("slot"):

    pack features -> fold weights (M, u) -> fused forward -> loss + cotangent -> fused backward
    -> weight gradients -> [gradient all-reduce over NCCL] -> Adam

On bounded-degree mesh batches (every mesh of the reference) all of that is ONE launch,
`gad_train_step_ell` (csrc/ell_kernels.cuh: k_ell_train): each CTA runs pack + forward + loss +
backward of its tiles out of shared memory and the last CTA to finish reduces the per-tile
partials in a fixed order, applies the chain rule to the Linear parameters, takes the Adam step
and refolds (M, u) for the next step.  With more than one rank the kernel stops after the chain
rule, NCCL all-reduces the flat gradient, and Adam + refold follow as two tiny kernels.

`ode_method='rk4'` trains the same way through `gad_train_step_ell_rk4` (k_ell_train with RK4 steps) where a
tile fits its nine rows per node (`gad_ell_rk4_train_supported`).  Larger tiles and meshes beyond one CTA run the
launch chain: forward, mesh loss, the RK4 backward of `functional.rk4_backward_resident`'s choice, weight
gradients, Adam.  The step sizes get no gradient through RK4, so `learn_step` is refused.

Sharding (SURVEY 8e): a batch is a disjoint union of meshes, so ranks take contiguous shards of
whole meshes with no data-path collective; the only exchange is the all-reduce of the flat
gradient (144 + L floats).  The mesh loss is a mean over ALL nodes of the global batch
(`F.l1_loss`, run_GNN.py:80-84): every rank scales its cotangent by 1/(count_local * world) and
the all-reduce sums.

The model's parameters are re-pointed at views of one flat buffer (as DDP buckets do), so the
kernels, the all-reduce and Adam all work on contiguous memory and `model.state_dict()` /
`load_state_dict()` keep working unchanged.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import torch
import torch.distributed as dist

from . import _lib, dp
from . import functional as GF
from .GNN import GNN


class _Slot:
    """Device-resident inputs, outputs and scratch of one batch."""
    pass


class DeformerTrainer:
    def __init__(self, model: GNN, lr: Optional[float] = None, weight_decay: Optional[float] = None,
                 betas=(0.9, 0.999), eps: float = 1e-8, loss_fn: Optional[str] = None,
                 process_group=None, use_cuda_graph: bool = True):
        self.model = model
        opt = model.opt
        self.opt = opt
        self.dev = model._device()
        self.lr = float(opt.get("lr", 1e-3) if lr is None else lr)
        self.wd = float(opt.get("decay", 0.0) if weight_decay is None else weight_decay)
        self.betas, self.eps = betas, eps
        # Options GNN.forward and the reference training loop honour but this fused step does not implement
        # raise instead of silently training something else (src/run_GNN.py:80-88,109-131; src/GNN.py:231-237).
        if loss_fn is None and opt.get("loss_type", "mesh_loss") != "mesh_loss":
            raise NotImplementedError(
                f"DeformerTrainer fuses the mesh loss (loss_type='mesh_loss', src/run_GNN.py:105-107); opt['loss_type']="
                f"{opt['loss_type']!r} trains through GNN.forward + autograd instead.  Pass loss_fn='l1' / 'mse' explicitly "
                "to train the mesh loss on such a preset")
        if getattr(model, "n_glob_used", 0) or opt.get("gnn_inc_glob_feat_f") or opt.get("gnn_inc_glob_feat_uu"):
            raise NotImplementedError("DeformerTrainer: global CNN features are trained through GNN.forward + autograd "
                                      "(the fused step does not update the CNN's parameters)")
        if opt.get("softmax_temp_type") == "learnable_a":
            raise NotImplementedError("DeformerTrainer: the learnable temperature is trained through GNN.forward + autograd")
        if opt.get("gnn_normalize", False):
            raise NotImplementedError("DeformerTrainer: gnn_normalize=True (per-batch f / max f, src/GNN.py:231-237) is "
                                      "only implemented on the GNN.forward path")
        if opt.get("gnn_dont_train", False):
            raise NotImplementedError("DeformerTrainer: gnn_dont_train=True skips the optimizer step (src/run_GNN.py:122-131); "
                                      "evaluate with GNN.forward instead")
        self.loss_kind = (opt.get("loss_fn", "l1") if loss_fn is None else loss_fn)
        if self.loss_kind not in ("l1", "mse"):
            raise NotImplementedError(f"DeformerTrainer: loss_fn={self.loss_kind!r} (the reference has 'l1' and 'mse', "
                                      "src/run_GNN.py:80-84)")
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.use_graph = use_cuda_graph
        self.L = int(opt["num_layers"])
        self.Lw = 1 if opt["share_conv"] else self.L
        self.C = int(opt["hidden_dim"])
        self.CE = model.CE
        self.dim = model.dim
        self.method = GF.METHODS[opt.get("ode_method", "euler")]
        if self.method == GF.METHOD_RK4 and opt["learn_step"]:
            raise NotImplementedError("learn_step with ode_method='rk4': the step sizes get no gradient through RK4")
        self._flatten_parameters()
        self.slots: List[_Slot] = []
        self.graphs: Dict[int, torch.cuda.CUDAGraph] = {}
        self.epoch_graphs: Dict[tuple, torch.cuda.CUDAGraph] = {}
        self.lib = _lib.load()
        # data parallel on one NVLink node: the training kernel all-reduces the gradient itself over
        # peer memory (dp.PeerExchange); otherwise NCCL between the train kernel and Adam
        self.rank = dist.get_rank(process_group) if self.world > 1 else 0
        self.peer = None
        self.loopback = opt.get("gad_peer_loopback")     # (world, rank): single-process self-test of the exchange
        if self.loopback is not None:
            if self.world != 1:
                raise ValueError("gad_peer_loopback is a single-process self-test option")
            self.world, self.rank = int(self.loopback[0]), int(self.loopback[1])
            self.peer = dp.PeerExchange.loopback(self.lib, self.flat.numel(), self.dev, self.world, self.rank)
        elif self.world > 1 and bool(opt.get("gad_peer_allreduce", True)) and self.dev.type == "cuda":
            self.peer = dp.PeerExchange(self.lib, self.flat.numel(), self.dev, group=process_group)
        self.fused_dp = self.peer is not None and self.peer.ok
        # programmatic dependent launch between the train kernels of consecutive steps (one launch per step)
        self.use_pdl = bool(opt.get("gad_pdl", True)) and (self.world == 1 or self.fused_dp)
        self._route_override = None     # dp_selfcheck: force the NCCL routes on slots that use the peer exchange
        self.stream = torch.cuda.Stream(device=self.dev)
        self.counter = torch.zeros(1, dtype=torch.int32, device=self.dev)   # last-CTA election of k_ell_train
        self.sync_weights()

    # ------------------------------------------------------------------------------------
    def _flatten_parameters(self):
        """flat = [Wq (Lw,C,C) | bq (Lw,C) | Wk (Lw,C,C) | bk (Lw,C) | steps (L, if learn_step)]."""
        m, Lw, C = self.model, self.Lw, self.C
        convs = [m.conv_layers[0]] if self.opt["share_conv"] else list(m.conv_layers)
        nW, nb = Lw * C * C, Lw * C
        nsteps = self.L if self.opt["learn_step"] else 0
        n = 2 * nW + 2 * nb + nsteps
        flat = torch.empty(n, dtype=torch.float32, device=self.dev)
        gflat = torch.zeros(n, dtype=torch.float32, device=self.dev)
        o = 0
        self.Wq = flat[o:o + nW].view(Lw, C, C); self.gWq = gflat[o:o + nW].view(Lw, C, C); o += nW
        self.bq = flat[o:o + nb].view(Lw, C); self.gbq = gflat[o:o + nb].view(Lw, C); o += nb
        self.Wk = flat[o:o + nW].view(Lw, C, C); self.gWk = gflat[o:o + nW].view(Lw, C, C); o += nW
        self.bk = flat[o:o + nb].view(Lw, C); self.gbk = gflat[o:o + nb].view(Lw, C); o += nb
        with torch.no_grad():
            for l, c in enumerate(convs):
                for view, gview, p in ((self.Wq, self.gWq, c.lin_query.weight), (self.bq, self.gbq, c.lin_query.bias),
                                       (self.Wk, self.gWk, c.lin_key.weight), (self.bk, self.gbk, c.lin_key.bias)):
                    view[l].copy_(p.detach().to(self.dev))
                    p.data = view[l]
                    p.grad = gview[l]
            if nsteps:
                self.tau = flat[o:o + nsteps]
                self.gtau = gflat[o:o + nsteps]
                for l, s in enumerate(m.steps):
                    self.tau[l:l + 1].copy_(s.detach().to(self.dev).reshape(1))
                    s.data = self.tau[l:l + 1]
                    s.grad = self.gtau[l:l + 1]
            else:
                self.tau = torch.full((self.L,), float(self.opt["time_step"]), dtype=torch.float32, device=self.dev)
                self.gtau = None
        self.flat, self.gflat = flat, gflat
        self.exp_avg = torch.zeros_like(flat)
        self.exp_avg_sq = torch.zeros_like(flat)
        self.step_count = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self.Mu = torch.empty((Lw, self.CE * self.CE + self.CE), dtype=torch.float32, device=self.dev)
        self.gMu = torch.empty_like(self.Mu)

    def broadcast_parameters(self, src: int = 0):
        dp.broadcast_flat(self.flat, src=src, group=self.pg)
        self.sync_weights()

    def sync_weights(self):
        """Refold (M, u) from the Linear parameters.  The one-launch step keeps `Mu == fold(params)` as an
        invariant (its tail refolds after Adam); call this after changing the parameters from outside
        (`load_state_dict`, manual edits)."""
        with torch.cuda.device(self.dev):
            torch.cuda.current_stream(self.dev).synchronize()
            with torch.cuda.stream(self.stream):
                _lib.check(self.lib.gad_prepare_weights(_lib.ptr(self.Wq), _lib.ptr(self.bq), _lib.ptr(self.Wk), self.Lw,
                                                        self.C, self.CE, self.model.inv_temp, _lib.ptr(self.Mu),
                                                        self.stream.cuda_stream), "gad_prepare_weights")

    def _train_desc(self, s: "_Slot", tail: int) -> "_lib.TrainDesc":
        """Descriptor of one `gad_train_step_ell` launch on slot `s` (include/gadapt.h: gad_train_desc)."""
        P, g = _lib.ptr, s.graph
        count = s.N * self.dim
        b1, b2 = self.betas
        d = _lib.TrainDesc()
        if g.tile_ptr is None:      # cluster-resident meshes (gad_train_step_cluster)
            d.ell_in, d.ell_out, d.tile_ptr, d.N = P(g.cl_in), P(g.cl_out), P(g.mesh_ptr), s.N
            d.T, d.max_tile_nodes, d.max_deg = len(g.mesh_sizes), max(g.mesh_sizes), g.cl_deg
        else:
            d.ell_in, d.ell_out, d.tile_ptr, d.N = P(g.ell_in), P(g.ell_out), P(g.ell_tile_ptr), s.N
            d.T, d.max_tile_nodes, d.max_deg = g.T, g.max_tile_nodes, g.ell_deg
        d.x_comp, d.f, d.uu, d.f_scale, d.uu_scale, d.target = P(s.x_comp), P(s.f), P(s.uu), None, None, P(s.target)
        d.dim, d.CE = self.dim, self.CE
        d.Mu, d.tau, d.Lw, d.L, d.C, d.inv_temp = P(self.Mu), P(self.tau), self.Lw, self.L, self.C, self.model.inv_temp
        d.loss_kind = 0 if self.loss_kind == "l1" else 1
        d.grad_scale, d.loss_scale = dp.local_grad_scale(count, s.count_global, world=self.world), 1.0 / count
        d.states, d.gMu, d.g_tau, d.loss, d.x_phys = P(s.states), P(self.gMu), P(self.gtau), P(s.loss), P(s.x_phys)
        d.workspace, d.workspace_bytes = P(s.bwd_ws), s.bwd_ws_bytes
        d.tail, d.counter = tail, P(self.counter)
        d.Wq, d.bq, d.Wk = P(self.Wq), P(self.bq), P(self.Wk)
        d.gWq, d.gbq, d.gWk, d.gbk = P(self.gWq), P(self.gbq), P(self.gWk), P(self.gbk)
        d.params, d.grads, d.exp_avg, d.exp_avg_sq = P(self.flat), P(self.gflat), P(self.exp_avg), P(self.exp_avg_sq)
        d.n_params = self.flat.numel()
        d.lr, d.beta1, d.beta2, d.eps, d.weight_decay, d.adam_grad_scale = self.lr, b1, b2, self.eps, self.wd, 1.0
        d.step = P(self.step_count)
        d.flags = 1 if (self.use_pdl and tail == 2) else 0      # GAD_TRAIN_PDL
        d.peer_timeout_ms = 0
        if self.fused_dp and tail == 2:
            d.rank, d.world, d.peers, d.peer_seq = self.rank, self.world, P(self.peer.ptrs), P(self.peer.seq)
            d.peer_timeout_ms = int(self.opt.get("gad_peer_timeout_ms", 10000))
        return d

    # ------------------------------------------------------------------------------------
    def add_batch(self, data) -> int:
        """Make `data` (host or device Batch) resident: build/cached graph, static input buffers,
        saved-state and scratch buffers.  Returns the slot id."""
        m, dev, lib = self.model, self.dev, self.lib
        s = _Slot()
        with torch.cuda.device(dev):
            s.graph = m._graph(data, dev, allow_uniform=True)      # the trainer never reads attention weights
            N = s.graph.N
            s.N = N
            f32 = dict(dtype=torch.float32, device=dev)
            xc = data.x_comp if data.x_comp.dim() == 2 else data.x_comp.unsqueeze(-1)
            # node inputs of a step live in ONE device buffer [target | f | uu | x_comp] (segments padded to
            # 16 bytes, the TMA staging granularity), so that a packed host batch travels in one copy.  x_comp
            # comes last: datasets on one shared mesh (`randg`, src/data.py:143: every sample has the same
            # computational mesh) send it once, and a step's copy is the [target | f | uu] prefix only.
            has_f, has_uu = bool(self.opt["gnn_inc_feat_f"]), bool(self.opt["gnn_inc_feat_uu"])
            seg = [N * self.dim, N if has_f else 0, N if has_uu else 0, N * self.dim]
            offs, o = [], 0
            for n in seg:
                offs.append(o)
                o += (n + 3) // 4 * 4
            s.in_offs, s.in_sizes = offs, seg
            s.inbuf = torch.zeros(o, **f32)
            s.target = s.inbuf[offs[0]:offs[0] + seg[0]].view(N, self.dim)
            s.f = s.inbuf[offs[1]:offs[1] + seg[1]] if has_f else None
            s.uu = s.inbuf[offs[2]:offs[2] + seg[2]] if has_uu else None
            s.x_comp = s.inbuf[offs[3]:offs[3] + seg[3]].view(N, self.dim)
            s.states = torch.empty((self.L, N, self.CE), **f32)
            s.x_phys = torch.empty((N, self.dim), **f32)
            s.g_out = torch.empty((N, self.dim), **f32)
            s.loss = torch.zeros(1, **f32)
            s.loss_ws = torch.empty(lib.gad_mesh_loss_workspace_bytes(N * self.dim), dtype=torch.uint8, device=dev)
            T = s.graph.T if s.graph.tile_ptr is not None else 0
            s.bwd_ws_bytes = max(lib.gad_deform_bwd_workspace_bytes(N, self.CE, T, self.L),
                                 lib.gad_ell_workspace_bytes(self.CE, T, self.L))
            s.bwd_ws = torch.empty(s.bwd_ws_bytes, dtype=torch.uint8, device=dev)
            streaming = T == 0 or self.opt.get("gad_force_stream", False)
            if streaming:
                s.graph.ensure_wide(self.CE)     # wide rows for the streaming ELL kernels, built outside any capture
            s.prefer_stream = None
            s.rk4_fused = s.rk4_resident = False
            if self.method == GF.METHOD_RK4:
                g = s.graph
                s.rk4_fused = bool(T and GF.use_ell(g, self.CE)
                                   and lib.gad_ell_rk4_train_supported(self.CE, g.max_tile_nodes, g.ell_deg))
                if not self._fused_ell(s):
                    # launch chain: the RK4 backward kernel is chosen (and wide rows built) here, outside any capture
                    s.rk4_resident = GF.rk4_backward_resident(g, self.CE, self.opt.get("gad_force_stream", False))
                    s.bwd_ws_bytes = max(s.bwd_ws_bytes, lib.gad_deform_bwd_wide_rk4_workspace_bytes(N, self.CE))
                    s.bwd_ws = torch.empty(s.bwd_ws_bytes, dtype=torch.uint8, device=dev)
            if (T == 0 and self.method == GF.METHOD_EULER and not self.opt.get("gad_no_cluster", False)
                    and s.graph.ensure_cluster(self.CE)):
                s.prefer_stream = bool(s.graph.stream_train_preferred(self.CE))   # decided outside any capture
                need = lib.gad_cluster_workspace_bytes(self.CE, len(s.graph.mesh_sizes), s.graph.cl_C, self.L)
                if need > s.bwd_ws_bytes:
                    s.bwd_ws_bytes = need
                    s.bwd_ws = torch.zeros(need, dtype=torch.uint8, device=dev)
            s.fwd_ws_bytes = lib.gad_deform_workspace_bytes(N, self.CE, self.method) if streaming else 0
            s.fwd_ws = torch.empty(max(s.fwd_ws_bytes, 16), dtype=torch.uint8, device=dev)
            s.h2d_bytes = 0
            # Data parallel: add_batch is COLLECTIVE (every rank adds its shard of the same global batch, in the
            # same order).  Two things are agreed here, once per slot and outside any capture:
            #  * the mean of the loss is over the nodes of the GLOBAL batch (F.l1_loss on the whole batch,
            #    src/run_GNN.py:80-84): the cotangent scale uses the summed count, so ragged shards weigh right;
            #  * the gradient route.  Whether a rank can run the one-launch kernel (whose tail all-reduces over
            #    peer memory) depends on ITS shard (degree, mesh sizes, policy); a rank spinning in the peer
            #    exchange while another calls NCCL would hang both, so the route is the MIN over the ranks.
            s.count_global = N * self.dim
            s.peer_route = False
            if self.loopback is not None:
                s.count_global, s.peer_route = N * self.dim * self.world, bool(self._one_launch_local(s))
            elif self.world > 1:
                mine = 1 if (self.fused_dp and self._one_launch_local(s)) else 0
                t = torch.tensor([N * self.dim, 1 - mine], dtype=torch.int64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.pg)
                t = t.cpu()
                s.count_global = int(t[0])
                s.peer_route = bool(int(t[1]) == 0)
        self.slots.append(s)
        sid = len(self.slots) - 1
        self.load_inputs(sid, data)
        return sid

    def _host_buffer(self, numel: int, write_combined: bool) -> torch.Tensor:
        """Pinned fp32 host buffer.  Write-combined pages come from the library (`gad_host_alloc`); the tensor is a view
        of that allocation, which lives as long as the trainer (released by `close()`)."""
        if not write_combined:
            return torch.zeros(numel, dtype=torch.float32).pin_memory()
        p = C.c_void_p()
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.gad_host_alloc(numel * 4, 1, C.byref(p)), "gad_host_alloc")
        self.__dict__.setdefault("_host_allocs", []).append(p)
        buf = torch.frombuffer((C.c_float * numel).from_address(p.value), dtype=torch.float32)
        buf.zero_()
        buf._gad_pinned = True
        return buf

    def pack_host(self, sid: int, data, with_x_comp: bool = True, write_combined: bool = False) -> torch.Tensor:
        """One pinned host buffer holding `data`'s node inputs in the layout of slot `sid`
        ([target | f | uu | x_comp]): `load_inputs` / `run_from_host` then move a batch host -> device
        with a single copy.  `with_x_comp=False` packs the per-sample prefix [target | f | uu] only, for
        datasets whose samples share one computational mesh (the slot keeps the x_comp it was given by
        `add_batch`; the caller asserts that it does not change -- checked here against the slot).
        `write_combined=True`: write-combined pinned pages (written once here, read only by the device)."""
        s = self.slots[sid]
        xc = data.x_comp if data.x_comp.dim() == 2 else data.x_comp.unsqueeze(-1)
        tg = data.x_phys if data.x_phys.dim() == 2 else data.x_phys.unsqueeze(-1)
        if not with_x_comp and not torch.equal(xc.to(torch.float32).cpu(), s.x_comp.cpu()):
            raise ValueError("pack_host(with_x_comp=False): this batch's x_comp differs from the slot's resident one")
        n_total = s.inbuf.numel() if with_x_comp else s.in_offs[3]
        buf = self._host_buffer(n_total, write_combined)
        parts = [tg, data.f_tensor if s.f is not None else None, data.uu_tensor if s.uu is not None else None,
                 xc if with_x_comp else None]
        for off, n, t in zip(s.in_offs, s.in_sizes, parts):
            if t is not None and n:
                buf[off:off + n].copy_(t.reshape(-1))
        return buf

    def _copy_inputs(self, s: "_Slot", data, skip_x_comp: bool = False) -> int:
        """Enqueue the host -> device copies of one batch on the current stream; returns the bytes.
        `skip_x_comp`: the slot's resident x_comp is this batch's (dataset on one shared mesh)."""
        if torch.is_tensor(data):                       # packed (pack_host): one copy (whole buffer or its prefix)
            s.inbuf[:data.numel()].copy_(data, non_blocking=True)
            return data.numel() * 4
        xc = data.x_comp if data.x_comp.dim() == 2 else data.x_comp.unsqueeze(-1)
        tg = data.x_phys if data.x_phys.dim() == 2 else data.x_phys.unsqueeze(-1)
        nbytes = 0
        if not skip_x_comp:
            s.x_comp.copy_(xc, non_blocking=True); nbytes += xc.numel() * 4
        s.target.copy_(tg, non_blocking=True); nbytes += tg.numel() * 4
        if s.f is not None:
            s.f.copy_(data.f_tensor, non_blocking=True); nbytes += data.f_tensor.numel() * 4
        if s.uu is not None:
            s.uu.copy_(data.uu_tensor, non_blocking=True); nbytes += data.uu_tensor.numel() * 4
        return nbytes

    def load_inputs(self, sid: int, data, non_blocking: bool = True):
        """Copy one batch's node features and target mesh (host, ideally pinned; a `Batch` or a buffer
        packed by `pack_host`) into the slot."""
        s = self.slots[sid]
        with torch.cuda.stream(self.stream):
            s.h2d_bytes = self._copy_inputs(s, data)
            if not non_blocking:
                self.stream.synchronize()
        return s.h2d_bytes

    # ------------------------------------------------------------------------------------
    def _issue(self, s: _Slot, stream_ptr: int, with_optimizer: bool = True, stage: str = "all"):
        """Enqueue the kernels of one training step on `stream_ptr` (captured or eager)."""
        lib, P, chk = self.lib, _lib.ptr, _lib.check
        g = s.graph
        CE, L, Lw, C_, dim = self.CE, self.L, self.Lw, self.C, self.dim
        tiles = g.tile_ptr is not None and not self.opt.get("gad_force_stream", False)
        inv_temp = self.model.inv_temp
        ell = self._fused_ell(s)
        cluster = (not ell) and self._cluster(s)
        if ell or cluster:
            # ONE launch per step (csrc/ell_kernels.cuh: k_ell_train): pack + forward + loss + backward per
            # tile, then the last CTA reduces, applies the chain rule and -- single GPU -- takes the Adam step
            # and refolds (M, u) for the next step.  Data parallel: all-reduce, Adam and refold follow.
            single = (self.world == 1 or (s.peer_route and self._route_override is None)) and with_optimizer
            if stage in ("all", "pre") and cluster:
                chk(lib.gad_train_step_cluster(C.byref(self._train_desc(s, 2 if single else 1)), g.cl_C, stream_ptr),
                    "gad_train_step_cluster")
            elif stage in ("all", "pre") and self.method == GF.METHOD_RK4:
                chk(lib.gad_train_step_ell_rk4(C.byref(self._train_desc(s, 2 if single else 1)), stream_ptr),
                    "gad_train_step_ell_rk4")
            elif stage in ("all", "pre"):
                chk(lib.gad_train_step_ell(C.byref(self._train_desc(s, 2 if single else 1)), stream_ptr),
                    "gad_train_step_ell")
            if stage in ("all", "post") and with_optimizer and not single:
                b1, b2 = self.betas
                chk(lib.gad_adam_step(P(self.flat), P(self.gflat), P(self.exp_avg), P(self.exp_avg_sq), self.flat.numel(),
                                      self.lr, b1, b2, self.eps, self.wd, 1.0, P(self.step_count), stream_ptr),
                    "gad_adam_step")
                chk(lib.gad_prepare_weights(P(self.Wq), P(self.bq), P(self.Wk), Lw, C_, CE, inv_temp, P(self.Mu),
                                            stream_ptr), "gad_prepare_weights")
            return
        if stage in ("all", "pre"):
            chk(lib.gad_prepare_weights(P(self.Wq), P(self.bq), P(self.Wk), Lw, C_, CE, inv_temp, P(self.Mu), stream_ptr),
                "gad_prepare_weights")
            chk(lib.gad_pack_features(P(s.x_comp), P(s.f), P(s.uu), None, None, s.N, dim, CE, P(s.states), stream_ptr),
                "gad_pack_features")
            wide = (not tiles) and g.ensure_wide(CE)      # streaming ELL kernels (csrc/stream_ell.cu)
            if wide:
                chk(lib.gad_deform_fwd_wide(P(g.wide_in), s.N, g.wide_deg, g.wide_reach, P(s.states), dim, CE, P(self.Mu), Lw, P(self.tau), L,
                                            self.method, P(s.x_phys), P(s.states), P(s.fwd_ws), s.fwd_ws_bytes, stream_ptr),
                    "gad_deform_fwd_wide")
            else:
                chk(lib.gad_deform_fwd(P(g.rowptr), P(g.col_walk), s.N, g.E, P(g.tile_ptr) if tiles else None,
                                       g.T if tiles else 0, g.max_tile_nodes, g.max_tile_edges, P(s.states), dim, CE,
                                       P(self.Mu), Lw, P(self.tau), L, self.method, P(s.x_phys), P(s.states), P(s.fwd_ws),
                                       s.fwd_ws_bytes, stream_ptr),
                    "gad_deform_fwd")
            chk(lib.gad_mesh_loss(P(s.x_phys), P(s.target), s.N * dim, 0 if self.loss_kind == "l1" else 1,
                                  dp.local_grad_scale(s.N * dim, s.count_global, world=self.world), P(s.loss), P(s.g_out),
                                  P(s.loss_ws),
                                  stream_ptr),
                "gad_mesh_loss")
            if self.method == GF.METHOD_RK4 and s.rk4_resident:
                chk(lib.gad_deform_bwd_ell_rk4(P(g.ell_in), P(g.ell_out), s.N, P(g.ell_tile_ptr), g.T, g.max_tile_nodes,
                                               g.ell_deg, P(s.states), P(s.g_out), dim, CE, P(self.Mu), None, Lw,
                                               P(self.tau), L, P(self.gMu), None, P(s.bwd_ws), s.bwd_ws_bytes, stream_ptr),
                    "gad_deform_bwd_ell_rk4")
            elif self.method == GF.METHOD_RK4:
                chk(lib.gad_deform_bwd_wide_rk4(P(g.wide_in), P(g.wide_out), s.N, g.wide_deg, P(s.states), P(s.g_out),
                                                dim, CE, P(self.Mu), Lw, P(self.tau), L, P(self.gMu), None, P(s.bwd_ws),
                                                s.bwd_ws_bytes, stream_ptr), "gad_deform_bwd_wide_rk4")
            elif wide:
                chk(lib.gad_deform_bwd_wide(P(g.wide_in), P(g.wide_out), s.N, g.wide_deg, P(s.states), P(s.g_out), dim, CE,
                                            P(self.Mu), Lw, P(self.tau), L, P(self.gMu), P(self.gtau), None, P(s.bwd_ws),
                                            s.bwd_ws_bytes, stream_ptr), "gad_deform_bwd_wide")
            else:
                chk(lib.gad_deform_bwd(P(g.rowptr), P(g.col_walk), P(g.t_rowptr), P(g.t_dst_walk), s.N, g.E,
                                       P(g.tile_ptr) if tiles else None, g.T if tiles else 0, g.max_tile_nodes,
                                       g.max_tile_edges, P(s.states), P(s.g_out), dim, CE, P(self.Mu), Lw, P(self.tau), L,
                                       P(self.gMu), P(self.gtau), None, P(s.bwd_ws), s.bwd_ws_bytes, stream_ptr),
                    "gad_deform_bwd")
            chk(lib.gad_weight_grads(P(self.Wq), P(self.bq), P(self.Wk), P(self.gMu), Lw, C_, CE, inv_temp, P(self.gWq),
                                     P(self.gbq), P(self.gWk), P(self.gbk), stream_ptr), "gad_weight_grads")
        if stage in ("all", "post") and with_optimizer:
            b1, b2 = self.betas
            chk(lib.gad_adam_step(P(self.flat), P(self.gflat), P(self.exp_avg), P(self.exp_avg_sq), self.flat.numel(),
                                  self.lr, b1, b2, self.eps, self.wd, 1.0, P(self.step_count), stream_ptr),
                "gad_adam_step")

    def _allreduce(self, s: Optional[_Slot] = None):
        """NCCL all-reduce of the flat gradient -- unless the train kernel of this slot does the
        exchange itself over peer memory (fused_dp on the one-launch path)."""
        if s is not None and s.peer_route and self._route_override is None:
            return
        if self._route_override == "nccl_ordered":
            dp.allreduce_flat_ordered(self.gflat, group=self.pg)
        else:
            dp.allreduce_flat(self.gflat, group=self.pg)

    def _fused_ell(self, s: _Slot) -> bool:
        """The step of this slot is the one-launch kernel k_ell_train (gad_train_step_ell / _rk4)."""
        g = s.graph
        tiles = g.tile_ptr is not None and not self.opt.get("gad_force_stream", False)
        return bool(tiles and GF.use_ell(g, self.CE) and not self.opt.get("gad_no_fused_train", False)
                    and (self.method == GF.METHOD_EULER or s.rk4_fused))

    def _cluster(self, s: _Slot) -> bool:
        """Meshes too large for one CTA run on the cluster-resident kernel (csrc/cl_kernels.cu, Euler only)."""
        g = s.graph
        if not (self.method == GF.METHOD_EULER and g.tile_ptr is None and g.cl_in is not None
                and not self.opt.get("gad_no_cluster", False) and not self.opt.get("gad_force_stream", False)):
            return False
        if s.prefer_stream is None:      # one or two very large meshes: the streaming chain uses all SMs
            s.prefer_stream = bool(g.stream_train_preferred(self.CE))
        return not s.prefer_stream

    def _one_launch(self, s: _Slot) -> bool:
        """The step of this slot is ONE kernel including the optimizer (single GPU, or every rank agreed on the
        in-kernel peer exchange for it)."""
        return self._one_launch_local(s) and (self.world == 1 or s.peer_route)

    def _one_launch_local(self, s: _Slot) -> bool:
        return self._fused_ell(s) or self._cluster(s)

    def close(self):
        """Drop the captured graphs and the peer mappings (call on every rank, after the last step)."""
        self.stream.synchronize()
        self.graphs.clear()
        self.epoch_graphs.clear()
        for p in self.__dict__.pop("_host_allocs", []):
            self.lib.gad_host_free(p)
        if self.peer is not None:
            if self.world > 1 and self.loopback is None:
                dist.barrier(group=self.pg)
            self.peer.close()
            self.peer = None
            self.fused_dp = False

    def capture(self, sid: int):
        """Capture the step of slot `sid` into a CUDA graph (gradient all-reduce included)."""
        s = self.slots[sid]
        with torch.cuda.device(self.dev):
            # warm up on the side stream (first-call attribute setting, NCCL communicator set-up)
            self.stream.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(self.stream):
                saved = [t.clone() for t in (self.flat, self.exp_avg, self.exp_avg_sq, self.step_count)]
                for _ in range(2):
                    self._issue(s, self.stream.cuda_stream, stage="pre")
                    self._allreduce(s)
                    self._issue(s, self.stream.cuda_stream, stage="post")
                for t, v in zip((self.flat, self.exp_avg, self.exp_avg_sq, self.step_count), saved):
                    t.copy_(v)
            self.stream.synchronize()
            self.sync_weights()
            self.stream.synchronize()
            self.check_peer(collective=True)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.stream):
                cs = torch.cuda.current_stream(self.dev).cuda_stream
                self._issue(s, cs, stage="pre")
                self._allreduce(s)
                self._issue(s, cs, stage="post")
            self.graphs[sid] = g

    def capture_epoch(self, sids, timed: bool = False) -> tuple:
        """Capture the steps of the resident batches `sids`, in order, into ONE CUDA graph.  On a single
        GPU every step is one kernel and consecutive kernels are linked by programmatic dependent
        launch: step k + 1 stages its inputs (TMA) while step k still computes, then waits for it.

        `timed=True` captures a second, instrumented graph of the same steps for benchmarks: a short device-side
        spin, an event record, the steps, an event record (external events = event-record NODES of the graph).
        `run_epoch(sids, timed=True)` replays it and `epoch_elapsed_ms(sids)` reads the device time between the two
        records: the steps' own time, without the latency of getting a graph launch from the host to the device."""
        key = tuple(int(s) for s in sids)
        if timed:
            key = ("timed",) + key
        if key in self.epoch_graphs:
            return key
        for sid in set(key[1:] if timed else key):   # warm-up / attribute set-up happens in the single-step capture
            if sid not in self.graphs:
                self.capture(sid)
        with torch.cuda.device(self.dev):
            self.stream.synchronize()
            self.check_peer(collective=True)
            g = torch.cuda.CUDAGraph()
            ev = None
            if timed:
                ev = (torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True))
            with torch.cuda.graph(g, stream=self.stream):
                cur = torch.cuda.current_stream(self.dev)
                cs = cur.cuda_stream
                if timed:
                    torch.cuda._sleep(200000)          # ~0.1 ms: the graph is fully resident before the first record
                    ev[0].record(cur)
                for sid in (key[1:] if timed else key):
                    s = self.slots[sid]
                    self._issue(s, cs, stage="pre")
                    self._allreduce(s)
                    self._issue(s, cs, stage="post")
                if timed:
                    ev[1].record(cur)
            self.epoch_graphs[key] = g
            if timed:
                self._epoch_events = getattr(self, "_epoch_events", {})
                self._epoch_events[key] = ev
        return key

    def epoch_elapsed_ms(self, sids) -> float:
        """Device time of the last `run_epoch(sids, timed=True)` (between the graph's two event-record nodes)."""
        key = ("timed",) + tuple(int(s) for s in sids)
        ev = self._epoch_events[key]
        ev[1].synchronize()
        return ev[0].elapsed_time(ev[1])

    def _touch_params(self):
        # the kernels update the parameters in place without bumping tensor version counters
        self.model._param_epoch = getattr(self.model, "_param_epoch", 0) + 1

    def run_epoch(self, sids, timed: bool = False):
        """One pass over the resident batches `sids` (one training step each) as a single graph replay.
        Returns the per-slot loss tensors (device; each holds the loss of that slot's LAST step)."""
        if not self.use_graph:
            return [self.step(sid) for sid in sids]
        key = self.capture_epoch(sids, timed=timed)
        self._touch_params()
        with torch.cuda.stream(self.stream):
            self.epoch_graphs[key].replay()
        return [self.slots[sid].loss for sid in (key[1:] if timed else key)]

    def step(self, sid: int):
        """One training step on the resident batch `sid` (asynchronous; loss stays on the device)."""
        self._touch_params()
        if self.use_graph:
            if sid not in self.graphs:
                self.capture(sid)
            with torch.cuda.stream(self.stream):
                self.graphs[sid].replay()
        else:
            with torch.cuda.stream(self.stream):
                s = self.slots[sid]
                self._issue(s, self.stream.cuda_stream, stage="pre")
                self._allreduce(s)
                self._issue(s, self.stream.cuda_stream, stage="post")
        return self.slots[sid].loss

    def step_from_host(self, sid: int, data) -> float:
        """End-to-end step: host (pinned) inputs -> device, train step, loss back to the host."""
        self.load_inputs(sid, data)
        loss = self.step(sid)
        with torch.cuda.stream(self.stream):
            out = loss.to("cpu", non_blocking=False)
        return float(out)

    def train_batch(self, data, ring: int = 3) -> torch.Tensor:
        """The body of the reference's training loop on the batch the loader just yielded --
        `optimizer.zero_grad(); out = model(data); loss = loss_fn(out, data.x_phys); loss.backward();
        optimizer.step()` (src/run_GNN.py:99-131, mesh loss) -- as: copy this batch's node inputs to a resident slot
        (copy stream), replay the slot's one-launch training step, return the loss (device tensor, asynchronous;
        valid until the slot comes round again, `ring` batches later).  So the reference's loop keeps its shape:

            for data in loader:                 # a fresh (ideally pinned) host Batch per iteration
                loss = trainer.train_batch(data)

        Slots are found by topology: batches of a dataset on one mesh (`opt['gad_shared_topology']`, the reference's
        `randg` data) share `ring` slots -- the graph is built once, no topology tensor crosses PCIe again; any other
        batch gets slots keyed on the identity of its `edge_index` (re-used when the same Batch object returns)."""
        m = self.model
        if bool(self.opt.get("gad_shared_topology", False)):
            ei = data.edge_index
            key = ("shared", tuple(ei.shape), int(data.x_comp.shape[0]), tuple(getattr(data, "mesh_sizes", ()) or ())[:4])
        else:
            key = ("id", id(data.edge_index), data.edge_index.data_ptr())
        rings = self.__dict__.setdefault("_rings", {})
        entry = rings.get(key)
        if entry is None:
            entry = {"sids": [], "next": 0, "keep": data.edge_index}
            rings[key] = entry
        if len(entry["sids"]) < ring:
            sid = self.add_batch(data)            # builds / finds the graph, allocates the slot, copies the inputs
            entry["sids"].append(sid)
            if self.use_graph:
                self.capture(sid)
            self.slots[sid]._free = torch.cuda.Event()
            self.slots[sid]._ready = torch.cuda.Event()
        else:
            sid = entry["sids"][entry["next"] % ring]
            s = self.slots[sid]
            if not hasattr(self, "_copy_stream"):
                self._copy_stream = torch.cuda.Stream(device=self.dev)
            cs = self._copy_stream
            with torch.cuda.stream(cs):
                cs.wait_event(s._free)                         # the slot's previous step has consumed its inputs
                s.h2d_bytes = self._copy_inputs(s, data, skip_x_comp=key[0] == "shared")
                s._ready.record(cs)
            with torch.cuda.stream(self.stream):
                self.stream.wait_event(s._ready)
        entry["next"] += 1
        loss = self.step(sid)
        with torch.cuda.stream(self.stream):
            self.slots[sid]._free.record(self.stream)
        return loss

    def _relay_descriptor(self, relay, batch_bytes: int, R: int):
        """`gad_pipeline_relay` for run_from_host(relay=(device, fraction)): a staging buffer and a stream on the other
        device (allocated once, this creates a context there), peer access both ways."""
        dev2, frac = int(relay[0]), float(relay[1])
        mine = self.dev.index if self.dev.index is not None else torch.cuda.current_device()
        if dev2 == mine or not (0.0 < frac < 1.0):
            raise ValueError("relay = (another visible device, fraction in (0, 1))")
        rest = int(batch_bytes * frac) // 256 * 256
        if rest <= 0:
            return None
        direct = batch_bytes - rest
        key = (dev2, rest, R)
        if getattr(self, "_relay_key", None) != key:
            _lib.check(self.lib.gad_enable_peer_access(mine, dev2), "gad_enable_peer_access")
            self._relay_staging = torch.empty(R * rest, dtype=torch.uint8, device=f"cuda:{dev2}")
            self._relay_stream = torch.cuda.Stream(device=dev2)
            torch.cuda.synchronize(dev2)
            self._relay_key = key
        d = _lib.PipelineRelay()
        d.device, d.direct_bytes = dev2, direct
        d.stream, d.staging, d.staging_stride = self._relay_stream.cuda_stream, self._relay_staging.data_ptr(), rest
        return d

    def run_from_host(self, host_batches, steps: int, native: Optional[bool] = None, relay=None) -> torch.Tensor:
        """Pipelined end-to-end training loop over host-resident (pinned) batches: the inputs of step
        k + 1 travel host -> device on a copy stream while step k computes, and every step's loss is
        read back device -> host asynchronously into pinned memory.  Slot k % R receives batch
        k % len(host_batches); needs R = len(self.slots) >= 2.  Returns the `steps` losses (host).

        With CUDA graphs and batches packed by `pack_host`, the loop itself runs in the C library
        (`gad_pipeline_run`, csrc/host_pipeline.cu: seven CUDA API calls per step, no Python); otherwise, or
        with `native=False`, the same schedule is issued from Python.

        `relay=(device, fraction)` (native loop only): that fraction of every batch reaches this GPU through another
        visible GPU -- host -> staging there over ITS path to host memory, then NVLink -- for boxes whose GPUs do not
        have equal host paths (gad_pipeline_run_relay; `dp.balance_host_paths` picks partner and fraction)."""
        R = len(self.slots)
        if R < 2:
            raise ValueError("run_from_host needs at least two resident slots (double buffering)")
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(device=self.dev)
            self._in_ready = [torch.cuda.Event() for _ in range(R)]
            self._slot_free = [torch.cuda.Event() for _ in range(R)]
        if getattr(self, "_loss_pin", None) is None or self._loss_pin.numel() < steps:
            self._loss_pin = torch.empty(max(steps, 1024), dtype=torch.float32).pin_memory()   # cudaHostAlloc is slow: once
        losses = self._loss_pin[:steps]
        cs, ms = self._copy_stream, self.stream
        packed = all(torch.is_tensor(b) and (b.is_pinned() or getattr(b, "_gad_pinned", False)) and b.dtype == torch.float32
                     for b in host_batches)
        pure = all(self._one_launch(s) for s in self.slots)      # the step's graph holds library kernels only
        if native is None:
            native = self.use_graph and packed and pure
        if native:
            if not (self.use_graph and packed):
                raise ValueError("the native pipeline needs use_cuda_graph=True and pinned buffers from pack_host")
            nb = len(host_batches)
            if len({b.numel() for b in host_batches}) != 1:
                raise ValueError("packed host batches must have one size")
            slots = (_lib.PipelineSlot * R)()
            for sid, s in enumerate(self.slots):
                if sid not in self.graphs:
                    self.capture(sid)
                slots[sid].dev_inputs = s.inbuf.data_ptr()
                slots[sid].bytes = host_batches[0].numel() * 4
                slots[sid].graph_exec = self.graphs[sid].raw_cuda_graph_exec()
                slots[sid].loss_dev = s.loss.data_ptr()
                s.h2d_bytes = host_batches[0].numel() * 4
            hosts = (C.c_void_p * nb)(*[b.data_ptr() for b in host_batches])
            self._touch_params()
            rdesc = self._relay_descriptor(relay, host_batches[0].numel() * 4, R) if relay is not None else None
            with torch.cuda.device(self.dev):
                if rdesc is None:
                    _lib.check(self.lib.gad_pipeline_run(slots, R, hosts, nb, int(steps), losses.data_ptr(),
                                                         ms.cuda_stream, cs.cuda_stream), "gad_pipeline_run")
                else:
                    _lib.check(self.lib.gad_pipeline_run_relay(slots, R, hosts, nb, int(steps), losses.data_ptr(),
                                                               ms.cuda_stream, cs.cuda_stream, C.byref(rdesc)),
                               "gad_pipeline_run_relay")
            self.check_peer()
            return losses
        if relay is not None:
            raise ValueError("relay needs the native pipeline (use_cuda_graph=True, buffers from pack_host)")
        cs.wait_stream(ms)
        nb = len(host_batches)

        def upload(k):
            sid = k % R
            s, data = self.slots[sid], host_batches[k % nb]
            with torch.cuda.stream(cs):
                if k >= R:
                    cs.wait_event(self._slot_free[sid])      # step k - R has consumed this slot's inputs
                s.h2d_bytes = self._copy_inputs(s, data)
                self._in_ready[sid].record(cs)

        upload(0)
        for k in range(steps):
            sid = k % R
            if k + 1 < steps:
                upload(k + 1)
            with torch.cuda.stream(ms):
                ms.wait_event(self._in_ready[sid])
            loss = self.step(sid)
            with torch.cuda.stream(ms):
                losses[k:k + 1].copy_(loss, non_blocking=True)
                self._slot_free[sid].record(ms)
        ms.synchronize()
        return losses

    def check_peer(self, collective: bool = False):
        """Raise if an in-kernel gradient exchange timed out (device error word, csrc/ell_kernels.cuh:
        peer_allreduce).  With `collective=True` (every rank calls it, e.g. before a capture) the launch
        sequence numbers of all ranks are compared as well: the exchange pairs launches by sequence number, so an
        asymmetric launch on one rank (a warm-up only it ran) would desynchronise the parity slots for good."""
        if self.peer is None or not self.fused_dp:
            return
        seq = self.peer.seq.cpu()
        if int(seq[1]) != 0:
            raise RuntimeError(
                f"rank {self.rank}: the in-kernel gradient all-reduce of exchange #{int(seq[1]) & 0xffffffff} timed out "
                f"(gad_peer_timeout_ms={int(self.opt.get('gad_peer_timeout_ms', 10000))}): a peer died, skipped a step or "
                "issued a different launch sequence.  The Adam step of that launch was skipped; the trainer cannot continue")
        if collective and self.world > 1 and self.loopback is None:
            mine = torch.tensor([int(seq[0])], dtype=torch.int64, device=self.dev)
            every = [torch.empty_like(mine) for _ in range(self.world)]
            dist.all_gather(every, mine, group=self.pg)
            vals = [int(v.item()) for v in every]
            if any(v != vals[0] for v in vals):
                raise RuntimeError(f"peer exchange sequence numbers differ across ranks: {vals} -- every rank must issue "
                                   "the same sequence of training launches")

    def dp_selfcheck(self, sids, steps: int = 16) -> dict:
        """Correctness check of the data-parallel step on the live job (collective; every rank calls it).

        From a snapshot of the current optimizer state, `steps` training steps over the resident batches `sids`
        are run three times -- (a) the route the trainer uses (the gradient all-reduce inside the train kernel
        over peer memory, where the slots agreed on it), (b) NCCL all-gather of the per-rank gradients followed by
        the same rank-ordered fp32 sum, Adam and refold as separate kernels, (c) plain `ncclAllReduce` -- and the
        state is restored afterwards.  Reported: the parameters of all ranks are bit-identical after (a); (a) and
        (b) agree bit for bit (same operands, same order: anything else is a bug in the exchange); the largest
        relative deviation of (a) from (c), whose reduction order is NCCL's own (equal at 2 ranks, rounding-level
        beyond).  The verdicts are MIN-reduced over the ranks, so every rank returns the same dict."""
        if self.world <= 1:
            return {"world": 1, "ranks_equal": True, "vs_nccl": "n/a (single rank)"}
        state = (self.flat, self.exp_avg, self.exp_avg_sq, self.step_count)
        self.stream.synchronize()
        saved = [t.clone() for t in state]

        def run(route):
            with torch.cuda.stream(self.stream):
                for t, v in zip(state, saved):
                    t.copy_(v)
            self.stream.synchronize()
            self.sync_weights()
            self._route_override = route
            try:
                with torch.cuda.stream(self.stream):
                    for k in range(steps):
                        s = self.slots[sids[k % len(sids)]]
                        self._issue(s, self.stream.cuda_stream, stage="pre")
                        self._allreduce(s)
                        self._issue(s, self.stream.cuda_stream, stage="post")
                self.stream.synchronize()
            finally:
                self._route_override = None
            self.check_peer()
            return self.flat.detach().clone()

        a = run(None)
        b = run("nccl_ordered")
        c = run("nccl")
        with torch.cuda.stream(self.stream):
            for t, v in zip(state, saved):
                t.copy_(v)
        self.stream.synchronize()
        self.sync_weights()
        self.stream.synchronize()
        every = [torch.empty_like(a) for _ in range(self.world)]
        dist.all_gather(every, a, group=self.pg)
        ranks_equal = all(bool(torch.equal(e, a)) for e in every)
        exact = bool(torch.equal(a, b))
        dev_c = float(((a - c).abs().max() / c.abs().max().clamp_min(1e-30)).item())
        moved = float((a - saved[0]).abs().max().item())
        verdict = torch.tensor([int(ranks_equal), int(exact), int(moved > 0)], dtype=torch.int32, device=self.dev)
        dist.all_reduce(verdict, op=dist.ReduceOp.MIN, group=self.pg)
        worst = torch.tensor([dev_c], dtype=torch.float64, device=self.dev)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX, group=self.pg)
        peer_slots = sum(1 for sid in sids if self.slots[sid].peer_route)
        return {"world": self.world, "steps": steps, "slots": len(sids), "slots_on_peer_route": peer_slots,
                "ranks_equal": bool(verdict[0].item()),
                "vs_nccl": "bit-exact" if bool(verdict[1].item()) else "DIFFERS",
                "nccl_route": "ncclAllGather of the per-rank gradients + rank-ordered fp32 sum, Adam and refold as "
                              "separate kernels",
                "vs_nccl_allreduce_max_rel": float(worst.item()),
                "parameters_moved": bool(verdict[2].item())}

    def synchronize(self):
        self.stream.synchronize()
        self.check_peer()
