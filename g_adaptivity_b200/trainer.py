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

Global CNN features (`gnn_inc_glob_feat_f / _uu` with channels that survive the encoder) train as a chain of library
kernels: CNN forward, the per-mesh bias offset du (csrc/glob_train.cu), the mesh-resident forward and backward with du,
the adjoint of du, CNN backward into the flat gradient, Adam over Linear and CNN parameters (`_issue_chain`).

`loss_type='pde_loss'` (the reference's Poisson preset, src/run_GNN.py:109-110: mse(FEM solution on the deformed mesh,
u_true_fine)) trains through the same chain with the loss stage FEM forward (gad_fem1d_fwd / gad_fem2d_fwd) ->
gad_pde_loss -> FEM backward, the kernels GNN.forward + autograd run for that loss, so a step reproduces the module
path's gradient bit for bit (in 2-D up to the last bit of the FEM backward, whose fp64 shared-memory atomics leave the
order of its sums open).  u_true_fine and the Gaussians of the right-hand side are segments of the slot's input
buffer.  Such slots need meshes of equal size on the mesh-resident ELL kernels and what the FEM kernels accept (2-D: up to
38 x 38, at most 16 Gaussians and 16 cells per vertex); `add_batch` raises otherwise.  An explicit `loss_fn` trains
the mesh loss instead.

`gnn_normalize=True` (f / torch.max(f), uu / torch.max(uu) over the batch, src/GNN.py:231-237) keeps the slot's route and
puts gad_batch_max in front of it: every step recomputes the maxima of the resident f / uu (a batch copied into the
slot is normalised by its own), MAX-all-reduced over the ranks, into the f_scale / uu_scale the kernels divide by.

`softmax_temp_type='learnable_a'` (a trainable temperature per weight set, src/GRAND_plus.py:152-154,328-329) trains
through the chain of library kernels: the temperatures join the flat vector after the steps, each step folds them into
the weights (gad_temp_fold: Mu / temp) and takes their gradient from the deformer's (gad_temp_fold_bwd).  k_ell_train
cannot: its tail refolds (M, u) with a constant temperature.  Such slots need the mesh-resident ELL kernels.

Neither option is trained together with global CNN features, and gnn_dont_train is refused: those raise
NotImplementedError and train through GNN.forward + autograd.

`loss_type='modular'` (the reference's Burgers preset, src/run_GNN.py:111-131: an outside function returns (loss,
x_grads) for the detached x_phys and the loop back-propagates sum(x_phys * x_grads)) is the cotangent mode:
`forward(sid)` runs the step's forward and returns the slot's x_phys, the caller computes x_grads, and
`step(sid, cotangent=x_grads)` copies it into the slot's target segment and replays the step, whose loss stage (loss
kind 2, include/gadapt.h) back-propagates exactly that cotangent on every route; `train_batch(data, grad_fn)` is the
loop body.  Steps cannot be issued ahead of the caller (run_epoch, run_from_host raise).  An explicit `loss_fn` trains
the mesh loss instead.

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
import math
from typing import Dict, List, Optional

import torch
import torch.distributed as dist

from . import _lib, dp
from . import functional as GF
from .GNN import GNN


def _ptr_array(tensors):
    """Host array of device pointers (the per-layer weight / bias arguments of gad_cnn_fwd / gad_cnn_bwd)."""
    return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


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
        loss_type = opt.get("loss_type", "mesh_loss")
        if loss_fn is None and loss_type not in ("mesh_loss", "pde_loss", "modular"):
            raise NotImplementedError(
                f"DeformerTrainer trains the mesh loss, the pde loss and the modular loss (src/run_GNN.py:105-131); "
                f"opt['loss_type']={opt['loss_type']!r} trains through GNN.forward + autograd instead.  Pass loss_fn='l1' / "
                "'mse' explicitly to train the mesh loss on such a preset")
        # loss_type='pde_loss': mse(FEM solution on the deformed mesh, u_true_fine), unless loss_fn asks for the mesh loss
        self.pde = loss_fn is None and loss_type == "pde_loss"
        # loss_type='modular': the caller's cotangent of x_phys (src/run_GNN.py:111-131), unless loss_fn asks for the
        # mesh loss
        self.cot = loss_fn is None and loss_type == "modular"
        # softmax_temp_type='learnable_a': one trainable temperature per weight set (src/GRAND_plus.py:152-154,328-329)
        self.learn_temp = opt.get("softmax_temp_type") == "learnable_a"
        # gnn_normalize: f / torch.max(f) and uu / torch.max(uu) over the batch (src/GNN.py:231-237)
        self.normalize = bool(opt.get("gnn_normalize", False))
        if getattr(model, "n_glob_used", 0) and (self.learn_temp or self.normalize):
            raise NotImplementedError("DeformerTrainer: global CNN features together with gnn_normalize=True or "
                                      "softmax_temp_type='learnable_a' train through GNN.forward + autograd")
        if opt.get("gnn_dont_train", False):
            raise NotImplementedError("DeformerTrainer: gnn_dont_train=True skips the optimizer step (src/run_GNN.py:122-131); "
                                      "evaluate with GNN.forward instead")
        self.loss_kind = "pde" if self.pde else "cot" if self.cot else (opt.get("loss_fn", "l1") if loss_fn is None else loss_fn)
        if not (self.pde or self.cot) and self.loss_kind not in ("l1", "mse"):
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
        # global CNN channels that survive the encoder's truncation; with none the model is a plain deformer and its
        # CNNs are never run (GNN.forward skips them too, so torch.optim.Adam never touches their parameters)
        self.n_g = int(getattr(model, "n_glob_used", 0))
        self._flatten_parameters()
        self.slots: List[_Slot] = []
        self.graphs: Dict[int, torch.cuda.CUDAGraph] = {}
        self.fwd_graphs: Dict[int, torch.cuda.CUDAGraph] = {}
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
        """flat = [Wq (Lw,C,C) | bq (Lw,C) | Wk (Lw,C,C) | bk (Lw,C) | steps (L, if learn_step) | temperatures (Lw, if
        learnable_a) | CNN f | CNN uu], the parameters of each global feature extractor in gad_cnn_bwd's order (w_0,
        b_0, w_1, ...), when n_g > 0."""
        m, Lw, C = self.model, self.Lw, self.C
        convs = [m.conv_layers[0]] if self.opt["share_conv"] else list(m.conv_layers)
        nW, nb = Lw * C * C, Lw * C
        nsteps = self.L if self.opt["learn_step"] else 0
        ntemp = Lw if self.learn_temp else 0
        cnn_specs, before = [], 0
        for name in (("f", "uu") if self.n_g else ()):
            ext = getattr(m, f"global_feature_extractor_cnn_{name}", None)
            if ext is None:
                continue
            # an extractor whose outputs the encoder truncates away still trains (zero gradient, weight decay), as the
            # module's cat + slice gives it; it is never run
            cnn_specs.append((name, ext, [p for c in ext.convs for p in (c.weight, c.bias)], self.n_g > before))
            before += ext.out_channels
        n = 2 * nW + 2 * nb + nsteps + ntemp + sum(p.numel() for _, _, ps, _ in cnn_specs for p in ps)
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
            o += nsteps
            self.temp = self.gtemp = None
            if ntemp:
                self.temp, self.gtemp = flat[o:o + ntemp], gflat[o:o + ntemp]
                for l, c in enumerate(convs):
                    p = c.sm_temp_a
                    self.temp[l:l + 1].copy_(p.detach().to(self.dev).reshape(1))
                    p.data = self.temp[l:l + 1].view(p.shape)
                    p.grad = self.gtemp[l:l + 1].view(p.shape)
            o += ntemp
            self.cnn = []
            for name, ext, ps, used in cnn_specs:
                o0, ws, bs = o, [], []
                for p in ps:
                    k = p.numel()
                    view = flat[o:o + k]
                    view.copy_(p.detach().to(self.dev).reshape(-1))
                    p.data = view.view(p.shape)
                    p.grad = gflat[o:o + k].view(p.shape)
                    (ws if p.dim() > 1 else bs).append(view)
                    o += k
                self.cnn.append({"name": name, "used": used, "g": gflat[o0:o], "Cm": ext.mid_channels,
                                 "Co": ext.out_channels, "L": len(ext.convs),
                                 "wp": _ptr_array(ws), "bp": _ptr_array(bs)})
        self.flat, self.gflat = flat, gflat
        self.exp_avg = torch.zeros_like(flat)
        self.exp_avg_sq = torch.zeros_like(flat)
        self.step_count = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self.Mu = torch.empty((Lw, self.CE * self.CE + self.CE), dtype=torch.float32, device=self.dev)
        self.gMu = torch.empty_like(self.Mu)
        # learnable temperature: the folded weights the deformer kernels run on (Mu / temp) and the cotangent of Mu
        self.Mu_eff = torch.empty_like(self.Mu) if ntemp else None
        self.gMu_base = torch.empty_like(self.Mu) if ntemp else None

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

    def _loss_args(self, s: "_Slot") -> tuple:
        """(loss kind, cotangent scale, loss scale) of the slot's mesh-loss stage (include/gadapt.h: loss_kind).  The
        cotangent mode's loss is the pseudo-loss sum <x_phys, c>: every rank passes the cotangent of its own shard
        unscaled, and the all-reduce sums to the gradient of the union batch's pseudo-loss."""
        if self.cot:
            return 2, 1.0, 1.0
        count = s.N * self.dim
        return (0 if self.loss_kind == "l1" else 1), dp.local_grad_scale(count, s.count_global, world=self.world), 1.0 / count

    def _train_desc(self, s: "_Slot", tail: int) -> "_lib.TrainDesc":
        """Descriptor of one `gad_train_step_ell` launch on slot `s` (include/gadapt.h: gad_train_desc)."""
        P, g = _lib.ptr, s.graph
        b1, b2 = self.betas
        d = _lib.TrainDesc()
        if g.tile_ptr is None:      # cluster-resident meshes (gad_train_step_cluster)
            d.ell_in, d.ell_out, d.tile_ptr, d.N = P(g.cl_in), P(g.cl_out), P(g.mesh_ptr), s.N
            d.T, d.max_tile_nodes, d.max_deg = len(g.mesh_sizes), max(g.mesh_sizes), g.cl_deg
        else:
            d.ell_in, d.ell_out, d.tile_ptr, d.N = P(g.ell_in), P(g.ell_out), P(g.ell_tile_ptr), s.N
            d.T, d.max_tile_nodes, d.max_deg = g.T, g.max_tile_nodes, g.ell_deg
        d.x_comp, d.f, d.uu, d.target = P(s.x_comp), P(s.f), P(s.uu), P(s.target)
        d.f_scale, d.uu_scale = P(s.f_scale), P(s.uu_scale)
        d.dim, d.CE = self.dim, self.CE
        d.Mu, d.tau, d.Lw, d.L, d.C, d.inv_temp = P(self.Mu), P(self.tau), self.Lw, self.L, self.C, self.model.inv_temp
        d.loss_kind, d.grad_scale, d.loss_scale = self._loss_args(s)
        d.states, d.gMu, d.g_tau, d.loss, d.x_phys = P(s.states), P(self.gMu), P(self.gtau), P(s.loss), P(s.x_phys)
        d.workspace, d.workspace_bytes = P(s.bwd_ws), s.bwd_ws_bytes
        d.tail, d.counter = tail, P(self.counter)
        d.Wq, d.bq, d.Wk = P(self.Wq), P(self.bq), P(self.Wk)
        d.gWq, d.gbq, d.gWk, d.gbk = P(self.gWq), P(self.gbq), P(self.gWk), P(self.gbk)
        d.params, d.grads, d.exp_avg, d.exp_avg_sq = P(self.flat), P(self.gflat), P(self.exp_avg), P(self.exp_avg_sq)
        d.n_params = self.flat.numel()
        d.lr, d.beta1, d.beta2, d.eps, d.weight_decay, d.adam_grad_scale = self.lr, b1, b2, self.eps, self.wd, 1.0
        d.step = P(self.step_count)
        # GAD_TRAIN_PDL.  Not on a normalised slot: the kernel reads f_scale / uu_scale while staging its inputs, before
        # it waits on its predecessor, which there is gad_batch_max (or the all-reduce of its result).  Nor in the
        # cotangent mode: the staged target is the cotangent the caller has just written, and no train kernel
        # precedes the step there (forward and the caller's loss come between)
        d.flags = 1 if (self.use_pdl and tail == 2 and not s.norm and not self.cot) else 0
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
            tile_nodes = None
            if self.n_g:          # the module's planning: one mesh per tile, so the bias offset is per tile
                sizes = m._mesh_sizes(data)
                if any(n != sizes[0] for n in sizes):
                    raise NotImplementedError("global CNN features need meshes of equal size in a batch")
                tile_nodes = int(sizes[0])
            s.graph = m._graph(data, dev, allow_uniform=True, tile_nodes=tile_nodes)   # the trainer never reads attention weights
            N = s.graph.N
            s.N = N
            s.glob = bool(self.n_g)
            s.pde = self.pde
            s.temp = self.learn_temp
            s.norm = self.normalize
            s.chain = s.glob or s.pde or s.temp      # the step is _issue_chain's chain of library kernels
            s.du = None
            if s.glob:
                self._check_glob_graph(s.graph)
            if s.temp and (self.opt.get("gad_force_stream", False) or not GF.use_ell(s.graph, self.CE)):
                # k_ell_train refolds (M, u) with a constant temperature in its tail; the chain runs on these kernels
                raise NotImplementedError("softmax_temp_type='learnable_a' trains on the mesh-resident ELL kernels (meshes "
                                          "that fit a CTA, bounded degree); train this batch through GNN.forward + autograd")
            if s.pde:
                self._pde_setup(s, data)
            f32 = dict(dtype=torch.float32, device=dev)
            # node inputs of a step live in ONE device buffer [target | f | uu | x_comp] (segments padded to
            # 16 bytes, the TMA staging granularity), so that a packed host batch travels in one copy.  x_comp
            # comes last: datasets on one shared mesh (`randg`, src/data.py:143: every sample has the same
            # computational mesh) send it once, and a step's copy is the [target | f | uu] prefix only.
            # the global feature extractors read f / uu from the same buffer.  A pde slot's target is u_true_fine,
            # followed by the Gaussians of the right-hand side: [u_true_fine | centers | scales | f | uu | x_comp].
            has_f = bool(self.opt["gnn_inc_feat_f"]) or any(r["name"] == "f" and r["used"] for r in self.cnn)
            has_uu = bool(self.opt["gnn_inc_feat_uu"]) or any(r["name"] == "uu" and r["used"] for r in self.cnn)
            segs = [("target", (N, self.dim), torch.float32)]
            if s.pde:
                segs = [("target", (s.B * s.Q,), torch.float32), ("centers", s.gauss_shape, s.gauss_dtype),
                        ("scales", s.gauss_shape, s.gauss_dtype)]
            segs += [("f", (N if has_f else 0,), torch.float32), ("uu", (N if has_uu else 0,), torch.float32),
                     ("x_comp", (N, self.dim), torch.float32)]
            seg = [math.prod(shape) * (2 if dt == torch.float64 else 1) for _, shape, dt in segs]     # fp32 words
            offs, o = [], 0
            for n in seg:
                offs.append(o)
                o += (n + 3) // 4 * 4
            s.in_offs, s.in_sizes = offs, seg
            s.inbuf = torch.zeros(o, **f32)
            # typed views of the segments, in buffer order (host parts of a batch: _input_parts)
            s.in_views = [s.inbuf[off:off + n].view(dt).view(shape)
                          for off, n, (_, shape, dt) in zip(offs, seg, segs)]
            views = {name: (v if n else None) for (name, _, _), n, v in zip(segs, seg, s.in_views)}
            s.target, s.f, s.uu, s.x_comp = views["target"], views["f"], views["uu"], views["x_comp"]
            s.centers, s.scales = views.get("centers"), views.get("scales")
            # gnn_normalize: [max f, max uu] of the batch, recomputed by every step (gad_batch_max)
            s.norm_max = torch.ones(2, **f32) if s.norm else None
            s.f_scale = s.norm_max[0:1] if s.norm and s.f is not None else None
            s.uu_scale = s.norm_max[1:2] if s.norm and s.uu is not None else None
            s.states = torch.empty((self.L, N, self.CE), **f32)
            s.x_phys = torch.empty((N, self.dim), **f32)
            s.g_out = torch.empty((N, self.dim), **f32)
            s.loss = torch.zeros(1, **f32)
            ws = lib.gad_pde_loss_workspace_bytes(s.B, s.Q) if s.pde else lib.gad_mesh_loss_workspace_bytes(N * self.dim)
            s.loss_ws = torch.empty(ws, dtype=torch.uint8, device=dev)
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
            if s.glob:
                self._add_glob_buffers(s, data)
            s.fwd_ws_bytes = lib.gad_deform_workspace_bytes(N, self.CE, self.method) if streaming else 0
            s.fwd_ws = torch.empty(max(s.fwd_ws_bytes, 16), dtype=torch.uint8, device=dev)
            with torch.cuda.stream(self.stream):
                s.h2d_bytes = self._copy_inputs(s, data)
            if s.pde:
                self._pde_check(s)
            # Data parallel: add_batch is COLLECTIVE (every rank adds its shard of the same global batch, in the
            # same order).  Two things are agreed here, once per slot and outside any capture:
            #  * the mean of the loss is over the nodes of the GLOBAL batch (F.l1_loss on the whole batch,
            #    src/run_GNN.py:80-84): the cotangent scale uses the summed count, so ragged shards weigh right;
            #  * the gradient route.  Whether a rank can run the one-launch kernel (whose tail all-reduces over
            #    peer memory) depends on ITS shard (degree, mesh sizes, policy); a rank spinning in the peer
            #    exchange while another calls NCCL would hang both, so the route is the MIN over the ranks.
            #  A pde slot's mean is over the B * Q solution values of the global batch.
            count = s.B * s.Q if s.pde else N * self.dim
            s.count_global = count
            s.peer_route = False
            if self.loopback is not None:
                s.count_global, s.peer_route = count * self.world, bool(self._one_launch_local(s))
            elif self.world > 1:
                mine = 1 if (self.fused_dp and self._one_launch_local(s)) else 0
                t = torch.tensor([count, 1 - mine], dtype=torch.int64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.pg)
                t = t.cpu()
                s.count_global = int(t[0])
                s.peer_route = bool(int(t[1]) == 0)
        self.slots.append(s)
        return len(self.slots) - 1

    def _check_glob_graph(self, g):
        """A batch with global CNN features runs on the mesh-resident ELL kernels, one mesh per tile (GNN.forward's
        planning); anything else raises as the module path does."""
        if (self.opt.get("gad_force_stream", False) or not GF.use_ell(g, self.CE) or g.mesh_sizes is None
                or g.T != len(g.mesh_sizes)):
            raise NotImplementedError("DeformerTrainer trains global CNN features on the mesh-resident ELL kernels only "
                                      "(meshes that fit a CTA); train larger batches through GNN.forward + autograd")
        if self.method == GF.METHOD_RK4 and not GF.rk4_backward_resident(g, self.CE):
            raise NotImplementedError("DeformerTrainer trains global CNN features with ode_method='rk4' on meshes that fit "
                                      "the mesh-resident RK4 backward only; train larger batches through GNN.forward + "
                                      "autograd")

    def _pde_setup(self, s: "_Slot", data):
        """Refusals, FEM tables and buffers of a pde slot (loss_type='pde_loss'), from the helpers GNN.forward uses."""
        m, g, dev = self.model, s.graph, self.dev
        if self.opt.get("gad_force_stream", False) or not GF.use_ell(g, self.CE):
            raise NotImplementedError("pde_loss training runs on the mesh-resident ELL kernels (meshes that fit a CTA, "
                                      "bounded degree); train this batch through GNN.forward + autograd")
        s.B, s.Nm = m._pde_batch_shape(data, g, s.N)
        if getattr(data, "u_true_fine_tensor", None) is None or getattr(data, "pde_params", None) is None:
            raise ValueError("loss_type='pde_loss' needs data.u_true_fine_tensor and data.pde_params (src/run_GNN.py:109-110)")
        s.topo = m._fem2d_topology(dev, s.Nm) if self.dim == 2 else None
        s.eval_pts, order = m._pde_eval_points(dev)
        s.order = None if order is None else order.to(torch.int32)
        s.Q = int(s.eval_pts[0].numel())
        if data.u_true_fine_tensor.numel() != s.B * s.Q:
            raise ValueError(f"u_true_fine_tensor has {data.u_true_fine_tensor.numel()} entries; the FEM solution of "
                             f"{s.B} meshes at {s.Q} evaluation points has {s.B * s.Q}")
        centers, _ = m._pde_params_to_tensors(data.pde_params, s.B, "cpu")
        s.gauss_shape, s.gauss_dtype, s.G = tuple(centers.shape), centers.dtype, int(centers.shape[1])
        s.K = int(self.opt.get("load_quad_points", 101))
        s.count_global = s.B * s.Q
        f32 = dict(dtype=torch.float32, device=dev)
        s.sol = torch.zeros((s.B, s.Q), **f32)
        s.g_sol = torch.zeros((s.B, s.Q), **f32)
        if self.dim == 2:
            s.coeffs = torch.zeros((s.B, s.Nm), **f32)
            s.u64 = torch.zeros((s.B, s.Nm), dtype=torch.float64, device=dev)
            s.cg_iters = torch.zeros(s.B, dtype=torch.int32, device=dev)

    def _pde_check(self, s: "_Slot"):
        """Run the loss stage of a pde slot once, eagerly, on the computational meshes: the FEM kernels refuse what
        they cannot solve (2-D meshes beyond 38 x 38, more than 16 Gaussians, a vertex in more than 16 cells) here,
        before any capture, rather than inside a CUDA graph."""
        with torch.cuda.stream(self.stream):
            self._issue_pde_loss(s, self.stream.cuda_stream, coords=s.x_comp)
        self.stream.synchronize()

    def _add_glob_buffers(self, s: "_Slot", data):
        """CNN grid map, workspace, per-mesh CNN outputs / cotangents and the bias offset of a slot."""
        f32 = dict(dtype=torch.float32, device=self.dev)
        B, N1 = len(s.graph.mesh_sizes), int(s.graph.mesh_sizes[0])
        s.B = B
        s.cnn_hw = (int(round(N1 ** 0.5)),) * 2 if self.dim == 2 else (1, N1)
        s.cnn_gather = self.model._cnn_grid_map(data, N1, self.dev)
        used = [r for r in self.cnn if r["used"]]
        s.cnn_ws_bytes = max(self.lib.gad_cnn_workspace_bytes(B, s.cnn_hw[0], s.cnn_hw[1], r["Cm"], r["Co"], r["L"])
                             for r in used)
        s.cnn_ws = torch.empty(s.cnn_ws_bytes, dtype=torch.uint8, device=self.dev)
        s.cnn_scale = {r["name"]: torch.zeros(1, **f32) for r in used}
        s.cnn_out = {r["name"]: torch.zeros((B, r["Co"]), **f32) for r in used}
        s.cnn_gout = {r["name"]: torch.zeros((B, r["Co"]), **f32) for r in used}
        s.du = torch.zeros((B, self.Lw, self.CE), **f32)

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

    def _input_parts(self, s: "_Slot", data, with_x_comp: bool = True) -> list:
        """Host tensors of `data` for the slot's input segments, in buffer order (None: the segment is not sent)."""
        xc = data.x_comp if data.x_comp.dim() == 2 else data.x_comp.unsqueeze(-1)
        if s.pde:
            first = [data.u_true_fine_tensor, *self.model._pde_params_to_tensors(data.pde_params, s.B, "cpu")]
        elif self.cot:          # the target segment takes the caller's cotangent (step(sid, cotangent=...))
            first = [None]
        else:
            first = [data.x_phys if data.x_phys.dim() == 2 else data.x_phys.unsqueeze(-1)]
        return first + [data.f_tensor if s.f is not None else None, data.uu_tensor if s.uu is not None else None,
                        xc if with_x_comp else None]

    def pack_host(self, sid: int, data, with_x_comp: bool = True, write_combined: bool = False) -> torch.Tensor:
        """One pinned host buffer holding `data`'s node inputs in the layout of slot `sid`
        ([target | f | uu | x_comp]; a pde slot's target is [u_true_fine | centers | scales]): `load_inputs` /
        `run_from_host` then move a batch host -> device with a single copy.  `with_x_comp=False` packs the
        per-sample prefix (everything but x_comp) only, for datasets whose samples share one computational mesh
        (the slot keeps the x_comp it was given by `add_batch`; the caller asserts that it does not change -- checked
        here against the slot).  `write_combined=True`: write-combined pinned pages (written once here, read only by
        the device)."""
        s = self.slots[sid]
        xc = data.x_comp if data.x_comp.dim() == 2 else data.x_comp.unsqueeze(-1)
        if not with_x_comp and not torch.equal(xc.to(torch.float32).cpu(), s.x_comp.cpu()):
            raise ValueError("pack_host(with_x_comp=False): this batch's x_comp differs from the slot's resident one")
        n_total = s.inbuf.numel() if with_x_comp else s.in_offs[-1]
        buf = self._host_buffer(n_total, write_combined)
        for off, n, view, t in zip(s.in_offs, s.in_sizes, s.in_views, self._input_parts(s, data, with_x_comp)):
            if t is not None and n:
                buf[off:off + n].view(view.dtype).copy_(t.reshape(-1))
        return buf

    def _copy_inputs(self, s: "_Slot", data, skip_x_comp: bool = False) -> int:
        """Enqueue the host -> device copies of one batch on the current stream; returns the bytes.
        `skip_x_comp`: the slot's resident x_comp is this batch's (dataset on one shared mesh)."""
        if torch.is_tensor(data):                       # packed (pack_host): one copy (whole buffer or its prefix)
            s.inbuf[:data.numel()].copy_(data, non_blocking=True)
            return data.numel() * 4
        nbytes = 0
        for n, view, t in zip(s.in_sizes, s.in_views, self._input_parts(s, data, with_x_comp=not skip_x_comp)):
            if t is not None and n:
                view.copy_(t.reshape(view.shape), non_blocking=True)
                nbytes += t.numel() * t.element_size()
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
        """Enqueue the kernels of one training step on `stream_ptr` (captured or eager).  stage 'fwd': the step's
        forward only (cotangent mode: what `forward(sid)` runs) -- the work before the deformer and the deformer
        forward on the same kernels and arithmetic, so its x_phys is the step's bit for bit."""
        if s.norm and stage in ("all", "pre", "fwd"):
            self._issue_batch_max(s, stream_ptr)
        if s.chain:
            return self._issue_chain(s, stream_ptr, with_optimizer, stage)
        lib, P, chk = self.lib, _lib.ptr, _lib.check
        g = s.graph
        CE, L, Lw, C_, dim = self.CE, self.L, self.Lw, self.C, self.dim
        tiles = g.tile_ptr is not None and not self.opt.get("gad_force_stream", False)
        inv_temp = self.model.inv_temp
        ell = self._fused_ell(s)
        cluster = (not ell) and self._cluster(s)
        if stage == "fwd" and (ell or cluster):
            # the forward of the one-launch kernel: same rows, inputs and folded weights (the step keeps Mu == fold(params))
            if cluster:
                chk(lib.gad_deform_fwd_cluster(P(g.cl_in), P(g.mesh_ptr), len(g.mesh_sizes), max(g.mesh_sizes), g.cl_deg,
                                               g.cl_C, s.N, P(s.x_comp), P(s.f), P(s.uu), P(s.f_scale), P(s.uu_scale), dim,
                                               CE, P(self.Mu), None, Lw, P(self.tau), L, self.method, P(s.x_phys),
                                               P(s.states), stream_ptr), "gad_deform_fwd_cluster")
            else:
                chk(lib.gad_deform_fwd_ell_raw(P(g.ell_in), s.N, P(g.ell_tile_ptr), g.T, g.max_tile_nodes, g.ell_deg,
                                               P(s.x_comp), P(s.f), P(s.uu), P(s.f_scale), P(s.uu_scale), dim, CE,
                                               P(self.Mu), None, Lw, P(self.tau), L, self.method, P(s.x_phys),
                                               P(s.states), stream_ptr), "gad_deform_fwd_ell_raw")
            return
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
        if stage in ("all", "pre", "fwd"):
            chk(lib.gad_prepare_weights(P(self.Wq), P(self.bq), P(self.Wk), Lw, C_, CE, inv_temp, P(self.Mu), stream_ptr),
                "gad_prepare_weights")
            chk(lib.gad_pack_features(P(s.x_comp), P(s.f), P(s.uu), P(s.f_scale), P(s.uu_scale), s.N, dim, CE,
                                      P(s.states), stream_ptr), "gad_pack_features")
            wide = (not tiles) and g.ensure_wide(CE)      # streaming ELL kernels (csrc/stream_ell.cu)
            if wide:
                chk(lib.gad_deform_fwd_wide(P(g.wide_in), s.N, g.wide_deg, g.wide_reach, P(s.states), dim, CE, P(self.Mu), None, 0, Lw,
                                            P(self.tau), L, self.method, P(s.x_phys), P(s.states), P(s.fwd_ws), s.fwd_ws_bytes, stream_ptr),
                    "gad_deform_fwd_wide")
            else:
                chk(lib.gad_deform_fwd(P(g.rowptr), P(g.col_walk), s.N, g.E, P(g.tile_ptr) if tiles else None,
                                       g.T if tiles else 0, g.max_tile_nodes, g.max_tile_edges, P(s.states), dim, CE,
                                       P(self.Mu), Lw, P(self.tau), L, self.method, P(s.x_phys), P(s.states), P(s.fwd_ws),
                                       s.fwd_ws_bytes, stream_ptr),
                    "gad_deform_fwd")
            if stage == "fwd":
                return
            kind, grad_scale, _ = self._loss_args(s)
            chk(lib.gad_mesh_loss(P(s.x_phys), P(s.target), s.N * dim, kind, grad_scale, P(s.loss), P(s.g_out),
                                  P(s.loss_ws), stream_ptr), "gad_mesh_loss")
            if self.method == GF.METHOD_RK4 and s.rk4_resident:
                chk(lib.gad_deform_bwd_ell_rk4(P(g.ell_in), P(g.ell_out), s.N, P(g.ell_tile_ptr), g.T, g.max_tile_nodes,
                                               g.ell_deg, P(s.states), P(s.g_out), dim, CE, P(self.Mu), None, Lw,
                                               P(self.tau), L, P(self.gMu), None, P(s.bwd_ws), s.bwd_ws_bytes, stream_ptr),
                    "gad_deform_bwd_ell_rk4")
            elif self.method == GF.METHOD_RK4:
                chk(lib.gad_deform_bwd_wide_rk4(P(g.wide_in), P(g.wide_out), s.N, g.wide_deg, P(s.states), P(s.g_out),
                                                dim, CE, P(self.Mu), None, 0, Lw, P(self.tau), L, P(self.gMu), None, None,
                                                P(s.bwd_ws), s.bwd_ws_bytes, stream_ptr), "gad_deform_bwd_wide_rk4")
            elif wide:
                chk(lib.gad_deform_bwd_wide(P(g.wide_in), P(g.wide_out), s.N, g.wide_deg, P(s.states), P(s.g_out), dim, CE,
                                            P(self.Mu), None, 0, Lw, P(self.tau), L, P(self.gMu), P(self.gtau), None, None,
                                            P(s.bwd_ws), s.bwd_ws_bytes, stream_ptr), "gad_deform_bwd_wide")
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

    def _issue_chain(self, s: _Slot, stream_ptr: int, with_optimizer: bool, stage: str):
        """The step of a slot that is not on the one-launch kernel, as a chain of library kernels on the mesh-resident
        ELL graph (a slot with global CNN features, a pde slot, or a learnable temperature):  [CNN forward -> bias
        offset du] -> [Mu / temp] -> deformer forward [with du] -> loss stage (mesh loss; or FEM forward -> pde loss ->
        FEM backward) -> deformer backward -> [temperature gradient, cotangent of Mu] -> weight gradients -> [adjoint of
        du (CNN cotangents and the du terms of gWq / gWk) -> CNN backward into the flat gradient] -> [all-reduce] ->
        Adam over the whole flat vector.  These are the kernels GNN.forward + autograd run for the same batch."""
        lib, P, chk = self.lib, _lib.ptr, _lib.check
        g, m = s.graph, self.model
        CE, L, Lw, C_, dim = self.CE, self.L, self.Lw, self.C, self.dim
        inv_temp = m.inv_temp
        Mu = self.Mu_eff if s.temp else self.Mu                    # the folded weights the deformer kernels run on
        gMu_w = self.gMu_base if s.temp else self.gMu              # the cotangent gad_weight_grads takes
        if s.glob:
            B = s.B
            used = [r for r in self.cnn if r["used"]]
            src = {"f": s.f, "uu": s.uu}
            H, W = s.cnn_hw
            g_f, g_uu = s.cnn_out.get("f"), s.cnn_out.get("uu")
            glob = (B, used[0]["Co"], self.n_g, P(self.Wq), P(self.Wk), Lw, C_, m.z_dim, m.live, CE, inv_temp)
        if stage in ("all", "pre", "fwd"):
            chk(lib.gad_prepare_weights(P(self.Wq), P(self.bq), P(self.Wk), Lw, C_, CE, inv_temp, P(self.Mu), stream_ptr),
                "gad_prepare_weights")
            if s.temp:
                chk(lib.gad_temp_fold(P(self.Mu), P(self.temp), Lw, CE, P(Mu), stream_ptr), "gad_temp_fold")
            if s.glob:
                for r in used:
                    u, scale = src[r["name"]], s.cnn_scale[r["name"]]
                    chk(lib.gad_absmax(P(u), u.numel(), P(scale), stream_ptr), "gad_absmax")
                    if self.world > 1 and self.loopback is None:       # the CNN normalises by the max over the GLOBAL batch
                        dist.all_reduce(scale, op=dist.ReduceOp.MAX, group=self.pg)
                    chk(lib.gad_cnn_fwd(P(u), P(s.cnn_gather), P(scale), B, H, W, r["Cm"], r["Co"], r["L"], r["wp"],
                                        r["bp"], P(s.cnn_out[r["name"]]), P(s.cnn_ws), s.cnn_ws_bytes, stream_ptr),
                        "gad_cnn_fwd")
                chk(lib.gad_glob_bias_fwd(P(g_f), P(g_uu), *glob, P(s.du), stream_ptr), "gad_glob_bias_fwd")
            # node features as GNN.forward feeds them (identity encoder: channels beyond CE are dropped)
            f = s.f if self.opt["gnn_inc_feat_f"] and dim < CE else None
            uu = s.uu if self.opt["gnn_inc_feat_uu"] and dim + (1 if f is not None else 0) < CE else None
            chk(lib.gad_deform_fwd_ell_raw(P(g.ell_in), s.N, P(g.ell_tile_ptr), g.T, g.max_tile_nodes, g.ell_deg,
                                           P(s.x_comp), P(f), P(uu), P(s.f_scale), P(s.uu_scale), dim, CE, P(Mu),
                                           P(s.du), Lw, P(self.tau), L, self.method, P(s.x_phys), P(s.states), stream_ptr),
                "gad_deform_fwd_ell_raw")
            if stage == "fwd":
                return
            if s.pde:
                self._issue_pde_loss(s, stream_ptr)
            else:
                kind, grad_scale, _ = self._loss_args(s)
                chk(lib.gad_mesh_loss(P(s.x_phys), P(s.target), s.N * dim, kind, grad_scale, P(s.loss), P(s.g_out),
                                      P(s.loss_ws), stream_ptr), "gad_mesh_loss")
            if self.method == GF.METHOD_RK4 and not s.rk4_resident:
                chk(lib.gad_deform_bwd_wide_rk4(P(g.wide_in), P(g.wide_out), s.N, g.wide_deg, P(s.states), P(s.g_out),
                                                dim, CE, P(Mu), None, 0, Lw, P(self.tau), L, P(self.gMu), None, None,
                                                P(s.bwd_ws), s.bwd_ws_bytes, stream_ptr), "gad_deform_bwd_wide_rk4")
            elif self.method == GF.METHOD_RK4:
                chk(lib.gad_deform_bwd_ell_rk4(P(g.ell_in), P(g.ell_out), s.N, P(g.ell_tile_ptr), g.T, g.max_tile_nodes,
                                               g.ell_deg, P(s.states), P(s.g_out), dim, CE, P(Mu), P(s.du), Lw,
                                               P(self.tau), L, P(self.gMu), None, P(s.bwd_ws), s.bwd_ws_bytes, stream_ptr),
                    "gad_deform_bwd_ell_rk4")
            else:
                chk(lib.gad_deform_bwd_ell(P(g.ell_in), P(g.ell_out), s.N, P(g.ell_tile_ptr), g.T, g.max_tile_nodes,
                                           g.ell_deg, P(s.states), P(s.g_out), dim, CE, P(Mu), P(s.du), Lw, P(self.tau),
                                           L, P(self.gMu), P(self.gtau), None, P(s.bwd_ws), s.bwd_ws_bytes, stream_ptr),
                    "gad_deform_bwd_ell")
            if s.temp:      # d loss / d temp into the flat gradient, and the cotangent of the base (M, u)
                chk(lib.gad_temp_fold_bwd(P(self.gMu), P(Mu), P(self.temp), Lw, CE, P(gMu_w), P(self.gtemp), stream_ptr),
                    "gad_temp_fold_bwd")
            chk(lib.gad_weight_grads(P(self.Wq), P(self.bq), P(self.Wk), P(gMu_w), Lw, C_, CE, inv_temp, P(self.gWq),
                                     P(self.gbq), P(self.gWk), P(self.gbk), stream_ptr), "gad_weight_grads")
            if s.glob:
                chk(lib.gad_glob_bias_bwd(P(g_f), P(g_uu), *glob, P(s.bwd_ws), s.bwd_ws_bytes, P(s.cnn_gout.get("f")),
                                          P(s.cnn_gout.get("uu")), P(self.gWq), P(self.gWk), stream_ptr),
                    "gad_glob_bias_bwd")
                for r in used:
                    u, scale = src[r["name"]], s.cnn_scale[r["name"]]
                    chk(lib.gad_cnn_bwd(P(u), P(s.cnn_gather), P(scale), B, H, W, r["Cm"], r["Co"], r["L"], r["wp"],
                                        r["bp"], P(s.cnn_gout[r["name"]]), P(r["g"]), P(s.cnn_ws), s.cnn_ws_bytes,
                                        stream_ptr), "gad_cnn_bwd")
        if stage in ("all", "post") and with_optimizer:
            b1, b2 = self.betas
            chk(lib.gad_adam_step(P(self.flat), P(self.gflat), P(self.exp_avg), P(self.exp_avg_sq), self.flat.numel(),
                                  self.lr, b1, b2, self.eps, self.wd, 1.0, P(self.step_count), stream_ptr),
                "gad_adam_step")

    def _issue_batch_max(self, s: _Slot, stream_ptr: int):
        """gnn_normalize: the maxima of the slot's resident f and uu into f_scale / uu_scale, the divisors the deformer
        kernels apply (f / torch.max(f), src/GNN.py:231-237).  Inside the step, so that every batch copied into the slot
        is normalised by its own maxima; with several ranks they are MAX-all-reduced to the global batch's."""
        for u, out in ((s.f, s.f_scale), (s.uu, s.uu_scale)):
            if out is not None:
                _lib.check(self.lib.gad_batch_max(_lib.ptr(u), u.numel(), _lib.ptr(out), stream_ptr), "gad_batch_max")
        if self.world > 1 and self.loopback is None:
            dist.all_reduce(s.norm_max, op=dist.ReduceOp.MAX, group=self.pg)

    def _issue_pde_loss(self, s: _Slot, stream_ptr: int, coords: Optional[torch.Tensor] = None):
        """Loss stage of a pde slot: FEM forward on the deformed meshes (`coords`, default the slot's x_phys) -> mean
        squared error of the solution against u_true_fine and its cotangent (gad_pde_loss) -> FEM backward into the
        cotangent of x_phys, s.g_out.  The kernels GNN.forward + autograd run for mse(sol, u_true_fine)."""
        lib, P, chk = self.lib, _lib.ptr, _lib.check
        x = s.x_phys if coords is None else coords
        grad_scale = 2.0 / float(s.count_global)         # torch's mse_loss backward over the global batch
        if self.dim == 2:
            t, (ex, ey) = s.topo, s.eval_pts
            fem = (P(t.cells), t.T, P(t.is_bc), s.Nm, P(t.star_cell), P(t.star_loc), t.D, P(x), P(s.centers),
                   P(s.scales), s.G, s.B, s.K, P(ex), P(ey), s.Q)
            chk(lib.gad_fem2d_fwd(*fem, P(s.coeffs), P(s.sol), P(s.u64), P(s.cg_iters), stream_ptr), "gad_fem2d_fwd")
            chk(lib.gad_pde_loss(P(s.sol), P(s.order), P(s.target), s.B, s.Q, grad_scale, P(s.loss), P(s.g_sol),
                                 P(s.loss_ws), stream_ptr), "gad_pde_loss")
            chk(lib.gad_fem2d_bwd(*fem, P(s.u64), P(s.g_sol), P(s.g_out), stream_ptr), "gad_fem2d_bwd")
        else:
            fem = (P(x), P(s.centers), P(s.scales), P(s.eval_pts[0]))
            chk(lib.gad_fem1d_fwd(*fem, s.B, s.Nm, s.G, s.K, s.Q, P(s.sol), None, stream_ptr), "gad_fem1d_fwd")
            chk(lib.gad_pde_loss(P(s.sol), None, P(s.target), s.B, s.Q, grad_scale, P(s.loss), P(s.g_sol),
                                 P(s.loss_ws), stream_ptr), "gad_pde_loss")
            chk(lib.gad_fem1d_bwd(*fem, P(s.g_sol), s.B, s.Nm, s.G, s.K, s.Q, P(s.g_out), stream_ptr), "gad_fem1d_bwd")

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
        return bool(tiles and not s.chain and GF.use_ell(g, self.CE) and not self.opt.get("gad_no_fused_train", False)
                    and (self.method == GF.METHOD_EULER or s.rk4_fused))

    def _cluster(self, s: _Slot) -> bool:
        """Meshes too large for one CTA run on the cluster-resident kernel (csrc/cl_kernels.cu, Euler only)."""
        g = s.graph
        if not (self.method == GF.METHOD_EULER and not s.chain and g.tile_ptr is None and g.cl_in is not None
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
        self.fwd_graphs.clear()
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
        self._refuse_cotangent_mode("capture_epoch")
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

    def _refuse_cotangent_mode(self, what: str):
        if self.cot:
            raise ValueError(f"{what}: with loss_type='modular' every step takes the cotangent of the x_phys of the current "
                             "parameters, so steps cannot be issued ahead of the caller's loss; use train_batch(data, "
                             "grad_fn) or forward(sid) -> step(sid, cotangent=x_grads)")

    def run_epoch(self, sids, timed: bool = False):
        """One pass over the resident batches `sids` (one training step each) as a single graph replay.
        Returns the per-slot loss tensors (device; each holds the loss of that slot's LAST step)."""
        self._refuse_cotangent_mode("run_epoch")
        if not self.use_graph:
            return [self.step(sid) for sid in sids]
        key = self.capture_epoch(sids, timed=timed)
        self._touch_params()
        with torch.cuda.stream(self.stream):
            self.epoch_graphs[key].replay()
        return [self.slots[sid].loss for sid in (key[1:] if timed else key)]

    def forward(self, sid: int) -> torch.Tensor:
        """Cotangent mode (loss_type='modular'): the forward of slot `sid`'s training step -- batch maxima, CNN
        features and bias offset, temperature fold where the slot has them, then the deformer -- on the step's kernels
        and arithmetic, so the step recomputes this x_phys bit for bit.  Returns the slot's static x_phys [N, dim]
        (device; valid until the next forward or step on the slot), ordered before later work on the caller's
        stream.  Captured as its own CUDA graph under use_cuda_graph."""
        if not self.cot:
            raise ValueError("forward(sid) is the cotangent mode of loss_type='modular'")
        s = self.slots[sid]
        with torch.cuda.device(self.dev):
            cur = torch.cuda.current_stream(self.dev)
            self.stream.wait_stream(cur)      # the caller is done with the previous x_phys
            if self.use_graph and sid not in self.fwd_graphs:
                with torch.cuda.stream(self.stream):      # warm-up: first-call attribute setting, communicators
                    self._issue(s, self.stream.cuda_stream, stage="fwd")
                self.stream.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=self.stream):
                    self._issue(s, torch.cuda.current_stream(self.dev).cuda_stream, stage="fwd")
                self.fwd_graphs[sid] = g
            with torch.cuda.stream(self.stream):
                if self.use_graph:
                    self.fwd_graphs[sid].replay()
                else:
                    self._issue(s, self.stream.cuda_stream, stage="fwd")
            cur.wait_stream(self.stream)
        return s.x_phys

    def _load_cotangent(self, s: _Slot, cot):
        """Copy the caller's cotangent of x_phys into the slot's target segment, on the trainer stream after the
        caller's current stream (where it was computed)."""
        if cot is None:
            raise ValueError("loss_type='modular': step(sid, cotangent=x_grads) needs the cotangent of forward(sid)'s x_phys")
        if not torch.is_tensor(cot) or cot.dtype != torch.float32 or tuple(cot.shape) != tuple(s.x_phys.shape):
            raise ValueError(f"the cotangent must be a float32 tensor of shape {tuple(s.x_phys.shape)}, got "
                             f"{(cot.dtype, tuple(cot.shape)) if torch.is_tensor(cot) else type(cot).__name__}")
        if cot.device.type == "cpu":
            if not cot.is_pinned():
                raise ValueError("a host cotangent must be in pinned memory")
        elif cot.device != s.x_phys.device:
            raise ValueError(f"the cotangent is on {cot.device}; the trainer runs on {s.x_phys.device}")
        with torch.cuda.device(self.dev):
            self.stream.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(self.stream):
                s.target.copy_(cot, non_blocking=True)
            if cot.is_cuda:
                cot.record_stream(self.stream)

    def step(self, sid: int, cotangent: Optional[torch.Tensor] = None):
        """One training step on the resident batch `sid` (asynchronous; loss stays on the device).

        Cotangent mode (loss_type='modular', no loss_fn): `cotangent` is required, the caller's x_grads for
        `forward(sid)`'s x_phys -- a float32 [N, dim] tensor on the trainer's device or pinned on the host.  It is
        copied into the slot, and the step recomputes its forward, back-propagates exactly that cotangent (the
        gradient of the pseudo-loss sum(x_phys * x_grads), src/run_GNN.py:111-131) and takes the Adam step; the loss
        it leaves is that pseudo-loss."""
        if self.cot:
            self._load_cotangent(self.slots[sid], cotangent)
        elif cotangent is not None:
            raise ValueError(f"step(cotangent=...) is the cotangent mode of loss_type='modular'; this trainer trains the "
                             f"{self.loss_kind!r} loss")
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
        self._refuse_cotangent_mode("step_from_host")
        self.load_inputs(sid, data)
        loss = self.step(sid)
        with torch.cuda.stream(self.stream):
            out = loss.to("cpu", non_blocking=False)
        return float(out)

    def train_batch(self, data, ring: int = 3, grad_fn=None):
        """The body of the reference's training loop on the batch the loader just yielded --
        `optimizer.zero_grad(); out = model(data); loss = loss_fn(out, data.x_phys); loss.backward();
        optimizer.step()` (src/run_GNN.py:99-131, mesh loss) -- as: copy this batch's node inputs to a resident slot
        (copy stream), replay the slot's one-launch training step, return the loss (device tensor, asynchronous;
        valid until the slot comes round again, `ring` batches later).  So the reference's loop keeps its shape:

            for data in loader:                 # a fresh (ideally pinned) host Batch per iteration
                loss = trainer.train_batch(data)

        Slots are found by topology: batches of a dataset on one mesh (`opt['gad_shared_topology']`, the reference's
        `randg` data) share `ring` slots -- the graph is built once, no topology tensor crosses PCIe again; any other
        batch gets slots keyed on the identity of its `edge_index` (re-used when the same Batch object returns).

        Cotangent mode (loss_type='modular'): `grad_fn(x_phys) -> (loss, x_grads)` is the reference's outside loss
        (src/run_GNN.py:111-131); the body is `forward(sid)` -> `grad_fn` -> `step(sid, cotangent=x_grads)`, and the
        return value is grad_fn's loss."""
        if self.cot != (grad_fn is not None):
            raise ValueError("train_batch(data, grad_fn) is the cotangent mode of loss_type='modular'" if self.cot else
                             "grad_fn is taken with loss_type='modular' only")
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
        if self.cot:
            loss, x_grads = grad_fn(self.forward(sid))
            self.step(sid, cotangent=x_grads)
        else:
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
        self._refuse_cotangent_mode("run_from_host")
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
        # the step's graph holds library kernels only (single GPU: a chain slot's chain of them; several ranks: no
        # collective in the graph, so not a normalised slot, whose maxima are all-reduced)
        pure = all((self._one_launch(s) and not (s.norm and self.world > 1 and self.loopback is None))
                   or (s.chain and self.world == 1) for s in self.slots)
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
