/*
 * gadapt.h -- C ABI of the B200 (sm_100a) g-adaptivity deformer hot path.
 *
 * Drop-in boundary for the GNN mesh-deformer of JRowbottomGit/g-adaptivity.  The reference has no
 * FFI of its own: its seam is the Python class surface `GNN(dataset, opt).forward(data)`
 * (src/GNN.py:144-306) and the operator `GRAND_plusConv.forward(x, edge_index, ...)`
 * (src/GRAND_plus.py:204-267).  These entry points are what a ctypes binding under that surface
 * calls (see INTEGRATION.md); the host-side mirror that does so lives in g_adaptivity_b200/.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name starts with `host_`;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that stream and
 *     performs no allocation and no host synchronisation (callers own all buffers, including
 *     the workspaces sized by the *_workspace_bytes queries);
 *   - return value 0 = OK, non-zero = error (message via gad_last_error(), thread-local);
 *   - no global mutable state: calls on distinct streams are re-entrant;
 *   - node-state tensors are row-major [N, CE] fp32 where CE (2, 4 or 8) is the number of live
 *     channels padded to a vector width.  With the reference's identity encoder
 *     (src/GNN.py:75-83) channels >= in_dim are exactly zero for the whole integration, so
 *     CE = pad(min(in_dim, hidden_dim)); the operator seam uses CE = hidden_dim.
 *   - the q/k projections of src/GRAND_plus.py:225-226 enter the kernels as the bilinear form
 *       s_e = <q_i, k_j> / (sqrt(C) T) = x_i^T M x_j + u^T x_j + (terms constant over the in-edges of i)
 *     with M = c Wq^T Wk, u = c Wk^T bq, c = 1/(sqrt(C) T); the row-constant terms cancel in the
 *     segment softmax (src/GRAND_plus.py:333), which is also why d/d(lin_key.bias) == 0.
 */
#ifndef GADAPT_H_
#define GADAPT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GAD_OK 0
#define GAD_ERR_ARG 1
#define GAD_ERR_CUDA 2
#define GAD_ERR_UNSUPPORTED 3

#define GAD_METHOD_EULER 0 /* x <- x + tau * F(x)          src/GNN.py:288-291                */
#define GAD_METHOD_RK4 1   /* one classical RK4 step of F per layer (extension, SURVEY A.1)  */

/* gad_graph_build writes this many int32 values to `info` */
#define GAD_INFO_WORDS 8
#define GAD_INFO_E 0            /* number of edges after filtering / loops               */
#define GAD_INFO_MAX_IN_DEG 1
#define GAD_INFO_MAX_OUT_DEG 2
#define GAD_INFO_CROSS_TILE 3   /* edges whose endpoints lie in different tiles (gad_graph_check_tiles) */
#define GAD_INFO_ELL_BAD 4      /* rows that do not fit the ELL form (gad_graph_build_ell)             */

int gad_version(void);
const char* gad_last_error(void);
/* Number of kernel launches this library has issued (or captured into a CUDA graph) so far. */
long long gad_launch_count(void);
/* Device properties the host-side planner needs (SM count, opt-in shared memory per block). */
int gad_device_info(int* host_sm_count, int* host_smem_optin_bytes, int* host_l2_bytes);

/* ---- K0: mesh-graph builder ------------------------------------------------------------
 * Replaces the per-call prologue of GNN.forward (src/GNN.py:206-223): boolean-mask filtering of
 * `edge_index`, appended corner self-loops, optional remove_self_loops + add_self_loops, and the
 * scatter/gather index structures PyG derives implicitly.  Produces
 *   filt_edge_index  int64 [2, Emax]  the edge list the reference's conv layers see, same order
 *   rowptr/col/eid   CSR by destination, rows in STABLE edge-list order (eid = edge position)
 *   t_rowptr/t_dst/t_slot  transpose (by source, stable) with the CSR slot of every edge
 * Emax = E0 + K + (self_loops ? N : 0).  The edge count E lands in info[GAD_INFO_E].
 * An edge e < E0 is dropped when any of the three masks is set (mask pointers may be NULL).
 * `extra_loops` are K node ids that each get one self-loop appended after the kept edges.
 */
size_t gad_graph_workspace_bytes(int64_t E0, int64_t K, int64_t N, int self_loops);
int gad_graph_build(const int64_t* edge_index, int64_t E0,
                    const uint8_t* mask_to_boundary, const uint8_t* mask_to_corner,
                    const uint8_t* mask_diff_boundary,
                    const int64_t* extra_loops, int64_t K, int self_loops, int64_t N,
                    int64_t* filt_edge_index, int32_t* rowptr, int32_t* col, int32_t* eid,
                    int32_t* t_rowptr, int32_t* t_dst, int32_t* t_slot, int32_t* info,
                    void* workspace, size_t workspace_bytes, void* stream);
/* Per-row ascending copy of a CSR (ptr = rowptr, idx = col) or CSC (t_rowptr, t_dst) index array:
 * the order in which the deformer kernels walk a row (bank-conflict-free gathers on structured
 * meshes).  The canonical, stable-ordered arrays are left untouched. */
int gad_graph_sort_rows(const int32_t* ptr, const int32_t* idx, int64_t N, int32_t* idx_sorted, void* stream);
/* Counts edges that leave their tile (tile_ptr int32 [T+1], node offsets) into info[GAD_INFO_CROSS_TILE]. */
int gad_graph_check_tiles(const int32_t* rowptr, const int32_t* col, int64_t N,
                          const int32_t* tile_ptr, int T, int32_t* info, void* stream);

/* Edge masks of firedrake_mesh_to_PyG (src/data.py:465-494) on the device.  edge_index int64 [2, E];
 * side_bits uint8 [N], bit k set when node v is on boundary marker k + 1 (src/data.py:451-455); outputs
 * uint8 [E]: to_boundary_edge_mask, to_corner_nodes_mask, diff_boundary_edges_mask.  Node ids outside
 * [0, N) are counted into info[7]. */
int gad_edge_masks(const int64_t* edge_index, int64_t E, const uint8_t* side_bits, int64_t N,
                   uint8_t* to_boundary, uint8_t* to_corner, uint8_t* diff_boundary, int32_t* info,
                   void* stream);

/* Content fingerprint of a (contiguous, 8-byte aligned) device buffer: out[0..1] += a 128-bit
 * position-sensitive hash of its bytes under `seed`.  The host keys its graph cache on the
 * fingerprints of edge_index / masks / batch, so that the FRESH Batch object the reference's loader
 * yields every iteration (src/run_GNN.py:97-105) finds the topology built for an earlier one. */
int gad_fingerprint(const void* data, size_t bytes, uint64_t seed, uint64_t* out, void* stream);

/* ---- weights ----------------------------------------------------------------------------
 * Mu[l] = { M (CE x CE, row-major, M[a][b]), u (CE) } for each of the Lw weight sets
 * (Lw = 1 when share_conv, src/GNN.py:131-137).  Wq/Wk are [Lw, C, C] ([out, in] like
 * torch Linear), bq [Lw, C].  Only the first min(CE, C) input columns are live.
 */
int gad_prepare_weights(const float* Wq, const float* bq, const float* Wk, int Lw, int C, int CE,
                        float inv_temp, float* Mu, void* stream);
/* Chain rule from (G_M, G_u) back to the Linear parameters; gbk is identically zero. */
int gad_weight_grads(const float* Wq, const float* bq, const float* Wk, const float* gMu, int Lw,
                     int C, int CE, float inv_temp, float* gWq, float* gbq, float* gWk, float* gbk,
                     void* stream);

/* ---- feature assembly (src/GNN.py:225-239 + identity encoder :75-83,270) -----------------
 * x0[i] = [x_comp[i, 0:dim], f[i] * f_scale, uu[i] * uu_scale, 0...] truncated/padded to CE.
 * f / uu may be NULL (feature switched off); *_scale may be NULL (= 1).
 */
int gad_pack_features(const float* x_comp, const float* f, const float* uu, const float* f_scale,
                      const float* uu_scale, int64_t N, int dim, int CE, float* x0, void* stream);

/* ---- deformer forward ---------------------------------------------------------------------
 * The whole of src/GNN.py:270-299: L layers of  x <- x + tau_l (A(x) x - x)  (or RK4 steps) and
 * the final slice to the first `dim` channels.  tau is a DEVICE array [L] (learn_step or not).
 * tile_ptr != NULL selects the mesh-resident kernel (one CTA per tile, state in shared memory
 * across all layers); tile_ptr == NULL selects the streaming kernels (one launch per F-eval).
 * states (optional) receives x^0 .. x^{L-1}  as [L, N, CE] for the backward.
 * workspace: gad_deform_workspace_bytes(N, CE, method) bytes (streaming path scratch).
 */
size_t gad_deform_workspace_bytes(int64_t N, int CE, int method);
int gad_deform_fwd(const int32_t* rowptr, const int32_t* col, int64_t N, int64_t E,
                   const int32_t* tile_ptr, int T, int max_tile_nodes, int max_tile_edges,
                   const float* x0, int dim, int CE, const float* Mu, int Lw, const float* tau, int L,
                   int method, float* x_phys, float* states, void* workspace, size_t workspace_bytes,
                   void* stream);

/* ---- deformer backward (Euler) ---------------------------------------------------------------
 * Cotangent g_xphys [N, dim] -> gMu [Lw, CE*CE+CE] (G_M, G_u), g_tau [L] (may be NULL),
 * g_x0 [N, CE] (may be NULL).  Deterministic: no floating-point atomics.
 * workspace: gad_deform_bwd_workspace_bytes(...) bytes.
 */
size_t gad_deform_bwd_workspace_bytes(int64_t N, int CE, int T, int L);
int gad_deform_bwd(const int32_t* rowptr, const int32_t* col, const int32_t* t_rowptr,
                   const int32_t* t_dst, int64_t N, int64_t E, const int32_t* tile_ptr, int T,
                   int max_tile_nodes, int max_tile_edges, const float* states,
                   const float* g_xphys, int dim, int CE, const float* Mu, int Lw, const float* tau,
                   int L, float* gMu, float* g_tau, float* g_x0, void* workspace,
                   size_t workspace_bytes, void* stream);

/* ---- streaming ELL ("wide") path: meshes too large for one CTA's shared memory, degree <= 7 ------
 * One launch per F-evaluation / backward pass like gad_deform_fwd / gad_deform_bwd without tiles, but
 * over rows  wide[i] = { int32 j_0 .. j_6, int32 valid }  (32 bytes; absolute neighbour ids, unused
 * slots = i, masked by `valid`): a node is ONE branch-free pass with no dependent index loads.
 * gad_graph_build_wide converts a (row-sorted) CSR or CSC; rows with more than 7 entries are counted
 * into info[GAD_INFO_ELL_BAD].  Workspaces: gad_deform_workspace_bytes / gad_deform_bwd_workspace_bytes.
 * `reach` = max |j - i| over the edges (the bandwidth of the node numbering), or -1 when unknown.  With a known
 * reach, and when all N / 256 CTAs with a window of (2 ceil(reach / 256) + 1) * 256 state rows in shared memory can
 * be co-resident, the forward runs ALL its F-evaluations in ONE cooperative launch (k_wide_persist: state in
 * registers, gathers from shared memory, halo rows exchanged through L2 as (value, epoch) pairs, no barrier);
 * same arithmetic, bit-identical results.  GAD_WIDE_PERSIST=0 in the environment keeps the launch chain. */
int gad_graph_build_wide(const int32_t* ptr, const int32_t* idx, int64_t N, void* wide_rows, int32_t* info,
                         void* stream);
/* Backward through classical RK4 steps on the streaming kernels (graphs without tiles, or tiles bypassed): from the
 * saved step inputs states [L, N, CE], per step three stage recomputes and four vjp passes of the Euler backward
 * kernels; cotangent g_xphys [N, dim] -> gMu [Lw, CE*CE+CE] (deterministic fixed-order reduction), g_x0 [N, CE] or
 * NULL.  No step-size gradient (as gad_deform_bwd_ell_rk4).  Replaces autograd through the reference's loop with an
 * RK4 step (north_star item 3; template classical_meshing/ma_mesh_1d.py:65-70). */
size_t gad_deform_bwd_wide_rk4_workspace_bytes(int64_t N, int CE);
int gad_deform_bwd_wide_rk4(const void* wide_in, const void* wide_out, int64_t N, int max_deg, const float* states,
                            const float* g_xphys, int dim, int CE, const float* Mu, int Lw, const float* tau, int L,
                            float* gMu, float* g_x0, void* workspace, size_t workspace_bytes, void* stream);
/* Largest node count the one-launch persistent forward takes on the current device for rows of this shape
 * (0: never -- reach unknown, window beyond 96 KB of shared memory, no cooperative launch). */
int64_t gad_wide_persist_nodes(int CE, int max_deg, int64_t reach);
int gad_deform_fwd_wide(const void* wide_in, int64_t N, int max_deg, int64_t reach, const float* x0, int dim, int CE,
                        const float* Mu, int Lw, const float* tau, int L, int method, float* x_phys,
                        float* states, void* workspace, size_t workspace_bytes, void* stream);
int gad_deform_bwd_wide(const void* wide_in, const void* wide_out, int64_t N, int max_deg, const float* states,
                        const float* g_xphys, int dim, int CE, const float* Mu, int Lw, const float* tau, int L,
                        float* gMu, float* g_tau, float* g_x0, void* workspace, size_t workspace_bytes,
                        void* stream);

/* ---- mesh-resident ELL path -------------------------------------------------------------------
 * The fast path for batches of bounded-degree meshes (every 1-D / 2-D mesh of the reference: in-
 * and out-degree <= 7 with self-loops).  Topology is one 16-byte row per node and direction:
 *     ell[i] = { uint16 off_0 .. off_6, uint16 valid },  off_q = (row_q - tile_start) * CE * 4
 * where bit q of `valid` says slot q holds a neighbour (the other slots point at some valid row of
 * the tile and are masked out).  Only the first W = {2,3,6,7} >= max_deg slots are used; WHICH slot
 * a neighbour sits in is free, and the builder picks one slot per neighbour offset (j - i) so that
 * on structured meshes consecutive nodes gather consecutive rows (no shared-memory bank conflicts).
 * Built once per graph by gad_graph_build_ell from the row-sorted CSR (ptr = rowptr, idx = col) or
 * CSC (t_rowptr, t_dst) arrays and the tile plan; rows that do not fit (degree > max_deg, neighbour
 * outside the tile, offset > 65535) are counted in info[GAD_INFO_ELL_BAD] and the caller must
 * fall back to gad_deform_fwd / gad_deform_bwd.  max_deg = max(in-degree, out-degree) of the graph.
 * gad_deform_fwd_ell / gad_deform_bwd_ell: same contract as gad_deform_fwd / gad_deform_bwd
 * (Euler or RK4 forward, Euler backward), CE in {2, 4}.
 * gad_deform_train_ell: the training pass of src/run_GNN.py:99-131 with loss_type = mesh_loss in ONE
 * launch per tile -- feature assembly (GNN.py:225-239), L Euler layers, mean L1 / MSE loss against
 * `target` [N, dim], and the backward -- followed by the fixed-order reduction:
 *     gMu [Lw, CE*CE+CE], g_tau [L] (may be NULL), loss[0] = loss_scale * sum |out - target| (or ^2),
 * with the cotangent grad_scale * d(sum)/d(out).  `states` [L, N, CE] is scratch (layer inputs),
 * x_phys [N, dim] is optional.  workspace: gad_ell_workspace_bytes(CE, T, L).
 *
 * PER-TILE BIAS OFFSET `du` [T, Lw, CE] (gad_deform_fwd_ell_raw, gad_deform_bwd_ell, gad_deform_bwd_ell_rk4; NULL =
 * none): added to the folded bias u of every node of the tile.  This is all the global CNN features of the
 * reference (src/GNN.py:242-268: a per-mesh constant vector appended to every node's features) do to the deformer:
 * constant channels stay constant under A(x) x - x, and in the logits x_i^T M x_j + u^T x_j every term they enter is
 * constant over the in-edges of i -- and cancels in the softmax -- except g^T M_gz z_j, a shift of u by M_gz^T g.
 * One mesh per tile is required (the caller plans tiles that way).  d loss / d du is read from the backward's
 * workspace, which begins with the per-tile partials [T, slots, CE*CE + CE + 1] (slots = L if Lw > 1 else 1):
 * entries CE*CE .. CE*CE + CE - 1 of a row are sum_i t_i = d loss / d u restricted to the tile.
 *
 * SHARED TOPOLOGY (tile_ptr == NULL, in every gad_*_ell entry point and in gad_train_desc): the batch is
 * T = ceil(N / max_tile_nodes) equal tiles of max_tile_nodes nodes (the last one may be shorter) and ell_in /
 * ell_out hold the rows of ONE tile (max_tile_nodes x 8 uint16), used by every tile.  This is the batch the
 * reference's `randg` datasets produce -- every sample lives on the same mesh (src/data.py:143), PyG's
 * collation only adds node offsets (a2) -- so the graph is built for one tile (O(mesh), not O(batch)) and
 * the per-step topology traffic is one table that stays in L2 / shared memory.
 */
int gad_graph_build_ell(const int32_t* ptr, const int32_t* idx, int64_t N, const int32_t* tile_ptr, int T,
                        int CE, int max_deg, void* ell_rows, int32_t* info, void* stream);
/* 1 when the ELL kernels can run tiles of this size (shared-memory fit), else 0. */
int gad_ell_supported(int CE, int max_tile_nodes, int max_deg, int train);
size_t gad_ell_workspace_bytes(int CE, int T, int L);
int gad_deform_fwd_ell(const void* ell_in, int64_t N, const int32_t* tile_ptr, int T, int max_tile_nodes,
                       int max_deg, const float* x0, int dim, int CE, const float* Mu, int Lw,
                       const float* tau, int L, int method, float* x_phys, float* states, void* stream);
/* The same forward from the RAW inputs of src/GNN.py:225-239 (x_comp [N, dim], f [N] | NULL, uu [N] |
 * NULL, optional batch-wide maxima f_scale / uu_scale): feature assembly + identity encoder are
 * fused into the kernel's input staging, so a deformer call is ONE launch.  `states` (optional,
 * [L, N, CE]) receives the layer inputs x^0 .. x^{L-1} for gad_deform_bwd_ell. */
int gad_deform_fwd_ell_raw(const void* ell_in, int64_t N, const int32_t* tile_ptr, int T, int max_tile_nodes,
                           int max_deg, const float* x_comp, const float* f, const float* uu,
                           const float* f_scale, const float* uu_scale, int dim, int CE, const float* Mu,
                           const float* du, int Lw, const float* tau, int L, int method, float* x_phys,
                           float* states, void* stream);
int gad_deform_bwd_ell(const void* ell_in, const void* ell_out, int64_t N, const int32_t* tile_ptr, int T,
                       int max_tile_nodes, int max_deg, const float* states, const float* g_xphys, int dim,
                       int CE, const float* Mu, const float* du, int Lw, const float* tau, int L, float* gMu,
                       float* g_tau, float* g_x0, void* workspace, size_t workspace_bytes, void* stream);
/* Backward through classical RK4 steps (the forward of gad_deform_fwd_ell* with method = GAD_METHOD_RK4; the
 * reference integrates with explicit Euler only, src/GNN.py:288-291 -- RK4 is this library's extension of the fused
 * ODE step, north_star item 3/4): gad_deform_bwd_ell's contract without g_tau.  Only the step inputs are read from
 * `states`; stage inputs are recomputed.  gad_ell_rk4_bwd_supported: 1 when a tile of that size fits the kernel's
 * shared memory (nine rows per node). */
int gad_deform_bwd_ell_rk4(const void* ell_in, const void* ell_out, int64_t N, const int32_t* tile_ptr, int T,
                           int max_tile_nodes, int max_deg, const float* states, const float* g_xphys, int dim,
                           int CE, const float* Mu, const float* du, int Lw, const float* tau, int L, float* gMu,
                           float* g_x0, void* workspace, size_t workspace_bytes, void* stream);
int gad_ell_rk4_bwd_supported(int CE, int max_tile_nodes, int max_deg);
/* One whole training step through classical RK4 steps in one launch: gad_train_step_ell's contract and descriptor
 * (declared below) with the forward of gad_deform_fwd_ell* (method = GAD_METHOD_RK4) and the backward of
 * gad_deform_bwd_ell_rk4 in the kernel; the loss and its cotangent are fused into stage 4 of the last step, and the
 * tail (reduction, chain rule, peer all-reduce, Adam, refold) is gad_train_step_ell's.  desc->g_tau must be NULL: the
 * step sizes get no gradient through RK4.  gad_ell_rk4_train_supported: 1 when a tile of that size fits the kernel's
 * shared memory (nine rows, the loss row and both ELL rows per node: 184 B at CE = 4); otherwise train through
 * gad_deform_fwd* + gad_mesh_loss + gad_deform_bwd_ell_rk4 / gad_deform_bwd_wide_rk4. */
struct gad_train_desc;
int gad_train_step_ell_rk4(const struct gad_train_desc* desc, void* stream);
int gad_ell_rk4_train_supported(int CE, int max_tile_nodes, int max_deg);
int gad_deform_train_ell(const void* ell_in, const void* ell_out, int64_t N, const int32_t* tile_ptr, int T,
                         int max_tile_nodes, int max_deg, const float* x_comp, const float* f,
                         const float* uu, const float* f_scale, const float* uu_scale, const float* target,
                         int dim, int CE, const float* Mu, int Lw, const float* tau, int L, int loss_kind,
                         float grad_scale, float loss_scale, float* states, float* gMu, float* g_tau,
                         float* loss, float* x_phys, void* workspace, size_t workspace_bytes, void* stream);

/* One WHOLE training step in one launch (src/run_GNN.py:99-131 with loss_type = mesh_loss): the
 * kernel of gad_deform_train_ell, whose last CTA to finish also runs the fixed-order reduction,
 * the chain rule to the Linear parameters (tail >= 1: what gad_weight_grads does) and -- tail == 2,
 * single-GPU training -- the Adam step on the flat parameter vector followed by the refold of
 * (M, u) for the NEXT step into Mu.  With tail == 1 the caller all-reduces `gWq..gbk` (data
 * parallel) and then calls gad_adam_step + gad_prepare_weights.  All pointers are device pointers.
 * `counter` is one zero-initialised uint32 owned by the caller (the kernel leaves it zero).
 * When the whole grid plus one CTA is resident at once, that extra CTA ("reducer") runs the tail:
 * it prepares while the tiles are processed and finishes once every tile CTA has checked in.
 * When tail == 2, Wq / bq / Wk must be views into `params` and gWq.. views into `grads`. */
typedef struct gad_train_desc {
    /* topology (gad_graph_build_ell) */
    const void* ell_in;
    const void* ell_out;
    const int32_t* tile_ptr;
    int64_t N;
    int32_t T, max_tile_nodes, max_deg;
    /* inputs: features of src/GNN.py:225-239 and the target mesh */
    const float* x_comp;
    const float* f;
    const float* uu;
    const float* f_scale;
    const float* uu_scale;
    const float* target;
    int32_t dim, CE;
    /* model */
    float* Mu;           /* [Lw, CE*CE+CE], current folded weights; rewritten when tail == 2 */
    const float* tau;    /* [L] */
    int32_t Lw, L, C;
    float inv_temp;
    /* loss: loss[0] = loss_scale * sum, cotangent = grad_scale * d(sum)/d(out) */
    int32_t loss_kind;
    float grad_scale, loss_scale;
    /* scratch and outputs */
    float* states;       /* [L, N, CE] */
    float* gMu;          /* [Lw, CE*CE+CE] */
    float* g_tau;        /* [L] or NULL */
    float* loss;         /* [1] */
    float* x_phys;       /* [N, dim] or NULL */
    void* workspace;     /* gad_ell_workspace_bytes(CE, T, L) */
    size_t workspace_bytes;
    /* tail */
    int32_t tail;        /* 1: reduce + weight grads, 2: + Adam + refold */
    uint32_t* counter;
    const float* Wq;
    const float* bq;
    const float* Wk;
    float* gWq;
    float* gbq;
    float* gWk;
    float* gbk;
    float* params;
    const float* grads;
    float* exp_avg;
    float* exp_avg_sq;
    int64_t n_params;
    float lr, beta1, beta2, eps, weight_decay, adam_grad_scale;
    int64_t* step;
    /* launch flags: bit 0 = programmatic dependent launch (the kernel may start while the previous
     * kernel of the stream is still running; it stages its inputs, then waits for it before touching
     * anything a kernel writes).  The inputs (x_comp, f, uu, target, ELL rows) must then not be
     * written by the preceding kernel of the stream. */
    int32_t flags;
    /* optional profiling aid: int64 [grid, 64] buffer receiving %globaltimer marks at the phase
     * boundaries of every CTA (NULL = off) */
    int64_t* trace;
    /* data parallel over peer memory (tail == 2, world > 1; see gad_peer_alloc): between the chain
     * rule and Adam the kernel stores its flat gradient into every rank's receive buffer over
     * NVLink and sums, in rank order, what the peers stored into its own -- the SUM all-reduce of
     * src/run_GNN.py's (single-process) gradient, fused into the step.  `peers` is a DEVICE array of
     * `world` receive-buffer pointers (entry `rank` = this rank's own buffer), `peer_seq` TWO
     * zero-initialised device uint32: [0] the launch sequence, advanced by one per launch (every rank
     * must issue the same sequence of launches), [1] an error word.  The wait for the peers' words is
     * bounded by `peer_timeout_ms` (0 = 10 000): when a contribution has not arrived by then (a peer
     * died, skipped a step or took the NCCL route) the kernel writes the failing sequence number into
     * peer_seq[1], skips the Adam step and the refold, and every later launch skips its wait as well;
     * the caller must check the word (it is sticky).  world <= 1 or peers == NULL: no exchange. */
    int32_t rank, world;
    void* const* peers;
    uint32_t* peer_seq;
    uint32_t peer_timeout_ms;
} gad_train_desc;
#define GAD_TRAIN_PDL 1
#define GAD_MAX_PEERS 16
int gad_train_step_ell(const gad_train_desc* desc, void* stream);

/* ---- cluster-resident training step: meshes beyond one CTA's shared memory (60x60 .. ~220x220) -------
 * One thread-block CLUSTER per mesh: the mesh is cut into `cluster_size` contiguous slabs, each kept
 * in one CTA's shared memory for the whole pass; rows of other slabs are read through distributed
 * shared memory.  gad_cluster_plan chooses the cluster size (2..16) and slab size for the largest
 * mesh; gad_graph_build_cluster converts a (row-sorted) CSR / CSC into cluster rows
 *     crow[i] = { u32 e_0 .. e_6, u32 valid },  e_q = (owner rank << 24) | (row offset in bytes)
 * (32 bytes per node); gad_train_step_cluster has gad_train_step_ell's contract with ell_in / ell_out
 * = cluster rows, tile_ptr = mesh_ptr [T + 1], T = meshes, max_tile_nodes = largest mesh, workspace of
 * gad_cluster_workspace_bytes.  Replaces src/run_GNN.py:99-131 for such meshes in one launch. */
int gad_cluster_plan(int CE, int max_mesh_nodes, int max_cluster /* <= 0: default (4) */, int* cluster_size,
                     int* slab_nodes);
int gad_graph_build_cluster(const int32_t* ptr, const int32_t* idx, const int32_t* mesh_ptr, int M,
                            int max_mesh_nodes, int CE, int cluster_size, void* rows, int32_t* info,
                            void* stream);
size_t gad_cluster_workspace_bytes(int CE, int M, int cluster_size, int L);
/* Planning aid: clusters of this shape the device can hold at once (cudaOccupancyMaxActiveClusters). */
int gad_cluster_occupancy(int CE, int cluster_size, int slab_nodes, int threads, int* max_active_clusters);
int gad_train_step_cluster(const gad_train_desc* desc, int cluster_size, void* stream);
/* Backward only (autograd of the module seam) from the states the forward saved: gad_deform_bwd_ell's
 * contract over cluster rows; workspace of gad_cluster_workspace_bytes. */
int gad_deform_bwd_cluster(const void* crows_in, const void* crows_out, const int32_t* mesh_ptr, int M,
                           int max_mesh_nodes, int max_deg, int cluster_size, int64_t N, const float* states,
                           const float* g_xphys, int dim, int CE, const float* Mu, int Lw, const float* tau, int L,
                           float* gMu, float* g_tau, float* g_x0, void* workspace, size_t workspace_bytes,
                           void* stream);
/* Forward only (module seam / inference), all L Euler layers or RK4 steps in ONE launch with the state
 * resident in the cluster's shared memory: gad_deform_fwd_ell_raw's contract over cluster rows. */
int gad_deform_fwd_cluster(const void* crows_in, const int32_t* mesh_ptr, int M, int max_mesh_nodes, int max_deg,
                           int cluster_size, int64_t N, const float* x_comp, const float* f, const float* uu,
                           const float* f_scale, const float* uu_scale, int dim, int CE, const float* Mu, int Lw,
                           const float* tau, int L, int method, float* x_phys, float* states, void* stream);

/* ---- operator seam: one GRAND_plusConv / GRAND_conv layer (src/GRAND_plus.py:204-267,380-382) --
 * res = A(x) x - x  for x [N, CE];  alpha (optional) [E] in filtered edge-list order.
 */
int gad_conv_fwd(const int32_t* rowptr, const int32_t* col, const int32_t* eid, int64_t N, int64_t E,
                 const float* x, int CE, const float* Mu, float* res, float* alpha, void* stream);
int gad_conv_bwd(const int32_t* rowptr, const int32_t* col, const int32_t* t_rowptr,
                 const int32_t* t_dst, int64_t N, int64_t E, const float* x, const float* g_res,
                 int CE, const float* Mu, float* gMu, float* g_x, void* workspace,
                 size_t workspace_bytes, void* stream);

/* ---- loss seam used by the training step (run_GNN.py:80-84,103-106): mean |out - target| or
 * mean (out - target)^2 over N*dim entries; writes the cotangent and a per-call loss scalar. */
int gad_mesh_loss(const float* out, const float* target, int64_t count, int kind /*0 l1, 1 mse*/,
                  float grad_scale, float* loss, float* g_out, void* workspace, void* stream);
size_t gad_mesh_loss_workspace_bytes(int64_t count);

/* ---- optimiser step on the flat parameter vector (run_GNN.py:88,128,131: torch.optim.Adam) ----
 * torch.optim.Adam semantics (L2 weight decay added to the gradient, bias-corrected moments).
 * `step` is a DEVICE int64 counter incremented by the kernel, so the call is CUDA-graph replayable.
 * grad_scale multiplies the gradient first (e.g. 1/world after a SUM all-reduce). */
int gad_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                  float lr, float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                  int64_t* step, void* stream);

/* ---- next row f1 (1-D): batched differentiable FEM solve after the deformer (loss_type = 'pde_loss') ----
 * Replaces the per-mesh Python loop of src/GNN.py:307-342 over torch_FEM_1D
 * (firedrake_difFEM/difFEM_1d.py:211-238: P1 stiffness matrix, load vector by `load_quad_points`-point
 * trapezoid quadrature of f = u''_true, Dirichlet values u_true(x_0), u_true(x_{n-1}), linear solve,
 * piecewise-linear interpolation at the Q evaluation points) and its autograd with respect to the mesh
 * points.  x [B, n] ascending mesh points per mesh, centers / scales [B, G] (Gaussians of u_true),
 * quad [Q] ascending.  fwd: sol [B, Q], coeffs [B, n-2] (may be NULL).  bwd: g_sol [B, Q] -> g_x [B, n]
 * (no gradient through the Dirichlet values, as difFEM_1d.py:221-222).  fp64 inside, fp32 outside. */
int gad_fem1d_fwd(const float* x, const float* centers, const float* scales, const float* quad, int B, int n, int G,
                  int load_quad_points, int Q, float* sol, float* coeffs, void* stream);
int gad_fem1d_bwd(const float* x, const float* centers, const float* scales, const float* quad, const float* g_sol,
                  int B, int n, int G, int load_quad_points, int Q, float* g_x, void* stream);

/* ---- next row f1 (2-D): batched differentiable FEM solve after the deformer on 2-D meshes ------------------
 * Replaces the per-mesh Python loop of src/GNN.py:327-335 over torch_FEM_2D
 * (firedrake_difFEM/difFEM_2d.py:345-372: P1 stiffness matrix from per-triangle gradients, Dirichlet rows,
 * load vector by torchquad's composite Simpson rule with `load_quad_points` points over the bounding box of
 * every node's star, linear solve, evaluation of sum_m coeffs_m phi_m at the Q evaluation points with the
 * edge / vertex repeat rule of `phim`) and its autograd with respect to the mesh points.  One topology per
 * batch: cells [T,3]; is_bc [N] (DirichletBC(V, 0, "on_boundary").nodes as a mask); star_cell / star_loc [N,D]
 * = cell id and local vertex index of the cells around every node in ascending cell order, -1 padded.
 * coords [B,N,2]; centers / scales [B,G,2] fp64 (as the reference passes them); eval_x / eval_y [Q].
 * fwd: coeffs [B,N], sol [B,Q], u64 [B,N] (fp64 coefficients kept for the backward), cg_iters [B] or NULL.
 * bwd: g_sol [B,Q] -> grad [B,N,2] (no gradient through Dirichlet values and cubature boxes, as :172, :298-309).
 * Parity against the reference's fixtures: tests/test_fem2d_gpu.py (B200), oracle/fem2d_host.cpp (host). */
int gad_fem2d_fwd(const int32_t* cells, int32_t T, const uint8_t* is_bc, int32_t N, const int32_t* star_cell,
                  const int32_t* star_loc, int32_t D, const float* coords, const double* centers, const double* scales,
                  int32_t G, int32_t B, int32_t load_quad_points, const float* eval_x, const float* eval_y, int32_t Q,
                  float* coeffs, float* sol, double* u64, int32_t* cg_iters, void* stream);
int gad_fem2d_bwd(const int32_t* cells, int32_t T, const uint8_t* is_bc, int32_t N, const int32_t* star_cell,
                  const int32_t* star_loc, int32_t D, const float* coords, const double* centers, const double* scales,
                  int32_t G, int32_t B, int32_t load_quad_points, const float* eval_x, const float* eval_y, int32_t Q,
                  const double* u64, const float* g_sol, float* grad, void* stream);

/* ---- peer memory for the data-parallel gradient exchange (one process per GPU, one node) -------
 * The reference trains single-process (src/run_GNN.py:95-131); sharding a batch by whole meshes
 * needs exactly one exchange per step, the SUM of the flat gradient.  gad_peer_alloc returns a
 * zeroed device buffer of gad_peer_exchange_bytes(world, n_params) and its CUDA IPC handle
 * (GAD_IPC_HANDLE_BYTES bytes, to be all-gathered by the host side); gad_peer_open maps a peer's
 * buffer from its handle.  gad_train_step_ell does the exchange inside the training kernel. */
#define GAD_IPC_HANDLE_BYTES 64
size_t gad_peer_exchange_bytes(int world, int64_t n_params);
int gad_peer_alloc(size_t bytes, void** dev_ptr, void* handle_out);
int gad_peer_open(const void* handle, void** dev_ptr);
int gad_peer_close(void* dev_ptr);
int gad_peer_free(void* dev_ptr);

/* ---- global CNN feature extractor (scope row f3) ----------------------------------------------------
 * GlobalFeatureExtractorCNN of src/feature_extractors.py:6-34 (wired at src/GNN.py:242-268):
 *     u / max|u|  ->  L x [conv kernel 3, stride 1, padding 1 + SELU]  ->  global average pool  ->  [B, Co]
 * on the H x W grid of one mesh's nodal values (Conv2d; H = 1: Conv1d over the W nodes of a 1-D mesh), one CTA per
 * mesh, all activation planes in shared memory.  u [B, H*W] mesh-major; `gather` [H*W] (or NULL) gives the node
 * whose value sits in grid cell y * W + x (the reordering of reshape_fd_tensor_to_grid, src/utils_data.py:125-141);
 * `scale` is one device float, max|u| over the batch.  weights / biases: HOST arrays of L device pointers in
 * torch's Conv layout [C_out, C_in, (3,) 3]: layer 0 is 1 -> Cm, layers 1 .. L-2 Cm -> Cm, layer L-1 Cm -> Co.
 * Backward: g_out [B, Co] -> g_params, flat in the order w_0, b_0, w_1, b_1, ... (gad_cnn_param_count entries);
 * the forward is recomputed, per-mesh parts are summed over the batch in fp64 in a fixed order (workspace of
 * gad_cnn_workspace_bytes; the same workspace size serves the forward).  When the L activation planes do not fit
 * the shared memory next to the other buffers (16 channels on a 30 x 30 grid) they live in the workspace instead
 * (L2-resident).  The grid values get no gradient.  Limits: L <= 8, channels <= 16. */
int64_t gad_cnn_param_count(int H, int Cm, int Co, int L);
size_t gad_cnn_workspace_bytes(int B, int H, int W, int Cm, int Co, int L);
int gad_cnn_fwd(const float* u, const int32_t* gather, const float* scale, int B, int H, int W, int Cm, int Co, int L,
                const float* const* weights, const float* const* biases, float* out, void* workspace,
                size_t workspace_bytes, void* stream);
int gad_cnn_bwd(const float* u, const int32_t* gather, const float* scale, int B, int H, int W, int Cm, int Co, int L,
                const float* const* weights, const float* const* biases, const float* g_out, float* g_params,
                void* workspace, size_t workspace_bytes, void* stream);

/* ---- host side of the end-to-end training loop ------------------------------------------------------
 * The reference's `for data in loader: ... loss.backward(); optimizer.step()` (src/run_GNN.py:95-131) with
 * the batches in PINNED host memory, as a double-buffered pipeline driven from C: for step k, slot
 * k % n_slots receives host batch k % n_host in ONE cudaMemcpyAsync on `copy_stream` (as soon as step
 * k - n_slots has released the slot), `compute_stream` waits for it, launches the slot's captured step
 * (`graph_exec`: a cudaGraphExec_t holding gad_train_step_ell on that slot) and copies the 4-byte loss
 * to losses_host[k] (pinned).  Blocks until the last step has finished.  n_slots >= 2. */
typedef struct gad_pipeline_slot {
    void* dev_inputs;        /* device buffer the packed batch is copied to */
    size_t bytes;            /* bytes per batch */
    void* graph_exec;        /* cudaGraphExec_t of this slot's training step */
    const float* loss_dev;   /* device scalar the step writes its loss to */
} gad_pipeline_slot;
int gad_pipeline_run(const gad_pipeline_slot* slots, int n_slots, const void* const* host_batches, int n_host,
                     int64_t steps, float* losses_host, void* compute_stream, void* copy_stream);
/* The same loop with a second path into the GPU (boxes whose GPUs do not have equal paths to host memory): the first
 * `direct_bytes` of every batch travel as above, the rest goes host -> `staging + slot * staging_stride` on ANOTHER
 * device (`device`, over that GPU's PCIe path, on `stream`, a stream of that device) and from there into the slot
 * over NVLink (cudaMemcpyPeerAsync; call gad_enable_peer_access first).  All of it inside the calling process.
 * relay == NULL: gad_pipeline_run. */
typedef struct gad_pipeline_relay {
    int device;              /* ordinal of the device the tail of each batch is relayed through */
    size_t direct_bytes;     /* bytes of each batch copied directly (multiple of 256) */
    void* stream;            /* cudaStream_t of `device` */
    void* staging;           /* buffer on `device`: n_slots * staging_stride bytes */
    size_t staging_stride;
} gad_pipeline_relay;
int gad_pipeline_run_relay(const gad_pipeline_slot* slots, int n_slots, const void* const* host_batches, int n_host,
                           int64_t steps, float* losses_host, void* compute_stream, void* copy_stream,
                           const gad_pipeline_relay* relay);
int gad_enable_peer_access(int dev_a, int dev_b);
/* Pinned host staging memory for packed batches (cudaHostAlloc); write_combined != 0 asks for write-combined pages:
 * written once by the host, read by the device without snooping the CPU caches. */
int gad_host_alloc(size_t bytes, int write_combined, void** host_ptr);
int gad_host_free(void* host_ptr);

#ifdef __cplusplus
}
#endif
#endif /* GADAPT_H_ */
