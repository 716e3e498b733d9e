// Mesh-resident ELL kernels: the whole multi-layer integration of a tile in ONE launch, and the
// whole training pass (forward, mesh loss, backward) of a tile in ONE launch.
//
// A batch is a disjoint union of meshes (PyG Batch semantics, SURVEY 8e), so a contiguous node
// range that does not split a mesh ("tile", planned on the host) is closed under the edge
// relation.  A CTA owns a tile at a time (persistent loop over tiles): the tile's node state lives
// in shared memory for all L layers (src/GNN.py:273-296) and HBM is touched only for the inputs,
// the saved layer states and the outputs.  Topology is the ELL form of ell_math.cuh (one 128-bit
// row per node and direction, byte offsets pre-multiplied), staged into shared memory by 1-D TMA
// bulk copies (cp.async.bulk + mbarrier) together with the initial state, or -- for tiles whose
// state alone fills the SM (50x50 meshes) -- streamed from L2 with a one-row software prefetch.
//
// Thread mapping: thread t owns nodes t, t + nthr, t + 2 nthr, ... of the tile, in every phase, so
// values a node carries between phases (gradient rows) are only ever touched by one thread and
// need no synchronisation; consecutive lanes own consecutive rows, which on row-major structured
// meshes makes the q-th neighbour gather of a warp hit consecutive shared-memory rows.
//
// Forward, per layer:    read X_cur (gathers), write X_nxt[i]          -> 1 barrier per layer
// Backward, per layer:   phase A (destination pass) reads X, writes GO / P / DL / GS[i]
//                        phase B (source pass) gathers GO / P / DL, writes GS[j], X[j] <- x^{l-1}
//                                                                      -> 2 barriers per layer
// Weight gradients: per-thread register accumulators, fixed-order block reduction, per-tile
// partials summed by a second tiny kernel.  No floating-point atomics: bit-reproducible.
#pragma once

#include <stdlib.h>

#include "common.cuh"
#include "ell_math.cuh"
#include "tail_math.cuh"

namespace gad {
namespace ell {

#ifndef GAD_ELL_MAXT
#define GAD_ELL_MAXT 512    // largest CTA; 1 CTA of 512 or 2 CTAs of 256 threads per SM: <= 128 registers, no spills
#endif
#ifndef GAD_ELL_MINB
#define GAD_ELL_MINB 1
#endif

// KIND_TRAIN_RK4: the rows of KIND_BWD_RK4, with the train tail's scratch rule of KIND_BWD.
enum Kind { KIND_FWD = 0, KIND_FWD_RK4 = 1, KIND_BWD = 2, KIND_BWD_RK4 = 3, KIND_TRAIN_RK4 = 4 };

constexpr size_t TAIL_SCRATCH_MIN = 24 * 1024;

struct Layout {
    uint32_t xa, xb, p, gs, dl, ein, eout, mu, red, bar, total;
    uint32_t y2, y3, y4, g, ab;   // RK4 backward: stage inputs, step cotangent, accumulated d/dy
};

__host__ __device__ inline Layout make_layout(int CE, int kind, int cap_nodes, bool ells, int nwarps) {
    Layout s{};
    size_t o = 0;
    auto bump = [&](size_t bytes) {
        const size_t at = o;
        o = (o + bytes + 127) & ~size_t(127);
        return (uint32_t)at;
    };
    const size_t rows = (size_t)cap_nodes * CE * sizeof(float);
    s.xa = bump(rows);
    s.xb = bump(rows);
    if (kind != KIND_FWD) {
        s.p = bump(rows);    // RK4: base state;   backward: p_i rows
        s.gs = bump(rows);   // RK4: accumulator;  backward: per-node gradient carry
    }
    const bool bwd = (kind == KIND_BWD || kind == KIND_BWD_RK4 || kind == KIND_TRAIN_RK4);
    const bool rk4_rows = (kind == KIND_BWD_RK4 || kind == KIND_TRAIN_RK4);
    if (bwd) s.dl = bump((size_t)cap_nodes * 8);
    if (rk4_rows) {
        s.y2 = bump(rows);
        s.y3 = bump(rows);
        s.y4 = bump(rows);
        s.g = bump(rows);
        s.ab = bump(rows);
    }
    if (ells) {
        s.ein = bump((size_t)cap_nodes * 16);
        if (bwd) s.eout = bump((size_t)cap_nodes * 16);
    }
    s.mu = bump((size_t)(CE * CE + CE) * sizeof(float));
    if (bwd) s.red = bump((size_t)(CE * CE + CE + 1) * nwarps * sizeof(float));
    if ((kind == KIND_BWD || kind == KIND_TRAIN_RK4) && o < TAIL_SCRATCH_MIN) o = TAIL_SCRATCH_MIN;   // train tail: [0, bar) is its scratch
    s.bar = bump(16);
    s.total = (uint32_t)o;
    return s;
}

struct Args {
    // topology
    const uint4* ell_in;
    const uint4* ell_out;
    const int32_t* tile_ptr;
    int T, cap_nodes;
    int64_t N;
    // model
    const float* Mu;
    const float* du;        // [T, Lw, CE] or null: per-tile offset of the folded bias u (global CNN features, GNN.py:242-268)
    const float* tau;
    int Lw, L, dim;
    // forward
    const float* x0;        // [N, CE] (forward kernel)
    float* x_phys;          // [N, dim] (may be null in the train kernel)
    float* states;          // [L, N, CE]: written by forward / train, read by backward / train
    // backward
    const float* g_xphys;   // [N, dim]
    float* partials;        // [T, slots, NACC]
    float* tau_partials;    // [T, L] or null
    float* g_x0;            // [N, CE] or null
    // train: fused feature assembly + loss
    const float* x_comp;
    const float* f;
    const float* uu;
    const float* f_scale;
    const float* uu_scale;
    const float* target;    // [N, dim]
    int loss_kind;          // 0: L1, 1: MSE, 2: target holds the caller's cotangent c of x_phys
    float grad_scale;       // cotangent = grad_scale * d|out - target| (or d(out - target)^2, or c)
    float* loss_partials;   // [T] sum over the tile of |d|, d^2 or out * c
    // train tail, run by the last CTA to finish (tail = 0: none, the host launches the reduction;
    // 1: reduction + weight gradients; 2: + Adam + the folded weights of the NEXT step)
    int tail;
    unsigned int* counter;  // zero before the first launch; the last CTA resets it
    float* gMu;             // [Lw, CE*CE+CE]
    float* g_tau;           // [L] or null
    float* loss;            // [1]
    float loss_scale;
    const float* Wq;        // [Lw, C, C] (views of `params` when tail == 2)
    const float* bq;
    const float* Wk;
    float* gWq;
    float* gbq;
    float* gWk;
    float* gbk;
    int C;
    float inv_temp;
    double cfold;           // tail::fold_scale(inv_temp, C), computed on the host
    float* Mu_next;         // = Mu (rewritten in place once every CTA is done with it)
    float* params;          // flat parameter vector and Adam state (tail == 2)
    const float* grads;
    float* exp_avg;
    float* exp_avg_sq;
    long long n_params;
    float lr, beta1, beta2, eps, weight_decay, adam_grad_scale;
    long long* step;
    int pdl;                // host side: launch with the programmatic-stream-serialization attribute
    int tail_cta;           // 1: the last CTA of the grid (an extra one, without tiles) runs the tail
    // data parallel over peer memory (tail == 2): receive buffers of all ranks, see peer.cu
    int rank, world;
    void* const* peers;
    unsigned int* peer_seq;   // [0] launch sequence, [1] error word (sequence of a timed-out exchange)
    unsigned long long peer_timeout_ns;
    long long* trace;       // optional [gridDim, 64] globaltimer marks of the train kernel (profiling aid)
};

// Phase timeline of the train kernel: thread 0 of every CTA stamps %globaltimer (ns) at the phase
// boundaries when Args::trace is set (scripts/ktrace.py); compiled out of the hot loops otherwise.
struct Tracer {
    long long* p;
    int n;
    __device__ __forceinline__ void mark() {
        if (p && threadIdx.x == 0 && n < 64) {
            long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            p[n++] = t;
        }
    }
};

template <int CE>
__device__ __forceinline__ Row<CE> load_row_cg(const float* base, int64_t i) {
    Row<CE> r;
    if constexpr (CE == 2) {
        const float2 t = __ldcg(reinterpret_cast<const float2*>(base + i * 2));
        r.v[0] = t.x;
        r.v[1] = t.y;
    } else {
        const float4 t = __ldcg(reinterpret_cast<const float4*>(base + i * CE));
        r.v[0] = t.x;
        r.v[1] = t.y;
        r.v[2] = t.z;
        r.v[3] = t.w;
    }
    return r;
}

template <int CE>
__device__ __forceinline__ void store_dims(float* __restrict__ out, int64_t i, int dim, const Row<CE>& r) {
    if (dim == 2) {
        *reinterpret_cast<float2*>(out + i * 2) = make_float2(r.v[0], r.v[1]);
    } else {
#pragma unroll
        for (int c = 0; c < CE; ++c)
            if (c < dim) out[i * dim + c] = r.v[c];
    }
}

template <int CE>
__device__ __forceinline__ Row<CE> load_dims(const float* __restrict__ in, int64_t i, int dim) {
    Row<CE> r;
    if (dim == 2) {
        const float2 t = *reinterpret_cast<const float2*>(in + i * 2);
        r.v[0] = t.x;
        r.v[1] = t.y;
#pragma unroll
        for (int c = 2; c < CE; ++c) r.v[c] = 0.f;
    } else {
#pragma unroll
        for (int c = 0; c < CE; ++c) r.v[c] = (c < dim) ? in[i * dim + c] : 0.f;
    }
    return r;
}

// Per-tile view of the ELL rows: shared memory (staged by TMA) or global memory (L2-resident).
template <bool ELLS>
struct EllView {
    const uint4* base;   // shared: tile-local rows; global: rows of the whole batch + n0
    __device__ __forceinline__ uint4 get(int i) const {
        if constexpr (ELLS) return base[i];
        else return __ldg(base + i);
    }
};

// Node range of a tile and the first ELL row of its table.  tile_ptr == nullptr is the SHARED-TOPOLOGY form: the
// batch consists of equal tiles of `cap_nodes` nodes (copies of one mesh, or of one group of meshes; the last
// tile may be shorter) that all use ONE table of tile-local ELL rows -- the reference's `randg` datasets put
// every sample on the same mesh (src/data.py:143), so the batch topology is one mesh's, B times.
__device__ __forceinline__ void tile_range(const Args& a, int tile, int& n0, int& NT, int& e0) {
    if (a.tile_ptr) {
        n0 = a.tile_ptr[tile];
        NT = a.tile_ptr[tile + 1] - n0;
        e0 = n0;
    } else {
        const long long first = (long long)tile * a.cap_nodes;
        const long long rest = a.N - first;
        n0 = (int)first;
        NT = rest < a.cap_nodes ? (int)rest : a.cap_nodes;
        e0 = 0;
    }
}

// Folded weights (M, u) of weight set `lw` into shared memory.  With per-mesh global features (row f3) the
// constant channels g of a mesh act on the attention only through a shift of u:  u_mesh = u + M_gz^T g  (the other
// terms are constant over the in-edges of a node and cancel in the softmax), handed in per tile as `du`.
template <int CE>
__device__ __forceinline__ void load_mu(const Args& a, float* Mu, int lw, int tile) {
    constexpr int MUSZ = CE * CE + CE;
    for (int t = threadIdx.x; t < MUSZ; t += blockDim.x) {
        float v = a.Mu[(size_t)lw * MUSZ + t];
        if (a.du && t >= CE * CE) v += a.du[((size_t)tile * a.Lw + lw) * CE + (t - CE * CE)];
        Mu[t] = v;
    }
}

// features = cat[x_comp, f, uu] (optionally f / max f, uu / max uu) + identity (zero-pad) encoder:
// src/GNN.py:225-239,75-83,270.  Inputs come from the TMA staging areas (`stage`) or from global
// memory; rows go to the shared-memory state buffer and, when `states0` is given, to states[0].
template <int CE>
__device__ __forceinline__ void assemble_rows(const Args& a, int n0, int NT, bool stage, const unsigned char* st_xc,
                                              const unsigned char* st_f, const unsigned char* st_uu, unsigned char* Xc,
                                              float* states0) {
    constexpr uint32_t RB = CE * sizeof(float);
    const int tid = threadIdx.x, nthr = blockDim.x;
    const float fs = (a.f && a.f_scale) ? a.f_scale[0] : 1.0f;
    const float us = (a.uu && a.uu_scale) ? a.uu_scale[0] : 1.0f;
    const int cf = a.dim, cu = a.dim + (a.f ? 1 : 0);
    for (int i = tid; i < NT; i += nthr) {
        const int64_t gi = (int64_t)n0 + i;
        Row<CE> x;
        float fv = 0.f, uv = 0.f;
        if (stage) {
            x = load_dims<CE>(reinterpret_cast<const float*>(st_xc), i, a.dim);
            if (a.f) fv = reinterpret_cast<const float*>(st_f)[i];
            if (a.uu) uv = reinterpret_cast<const float*>(st_uu)[i];
        } else {
            x = load_dims<CE>(a.x_comp, gi, a.dim);
            if (a.f) fv = a.f[gi];
            if (a.uu) uv = a.uu[gi];
        }
        if (a.f_scale) fv = fv / fs;     // the reference divides (f / torch.max(f), GNN.py:232)
        if (a.uu_scale) uv = uv / us;
#pragma unroll
        for (int c = 0; c < CE; ++c) {
            if (a.f && c == cf) x.v[c] = fv;
            if (a.uu && c == cu) x.v[c] = uv;
        }
        sts_row<CE>(Xc, i * RB, x);
        if (states0) store_row<CE>(states0, gi, x);
    }
}

// ============================================================================================
// forward
// ============================================================================================
template <int CE, int W, bool ELLS, int METHOD>
__global__ void __launch_bounds__(GAD_ELL_MAXT, GAD_ELL_MINB) k_ell_fwd(const Args a) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const Layout lay = make_layout(CE, METHOD == GAD_METHOD_RK4 ? KIND_FWD_RK4 : KIND_FWD, a.cap_nodes, ELLS,
                                   (nthr + 31) >> 5);
    unsigned char* Xc = smem + lay.xa;
    unsigned char* Xn = smem + lay.xb;
    unsigned char* XB = smem + lay.p;    // RK4 only
    unsigned char* AC = smem + lay.gs;   // RK4 only
    float* Mu = reinterpret_cast<float*>(smem + lay.mu);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + lay.bar);
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    uint32_t parity = 0;
    const size_t state_stride = (size_t)a.N * CE;

    for (int tile = blockIdx.x; tile < a.T; tile += gridDim.x) {
        int n0, NT, e0;
        tile_range(a, tile, n0, NT, e0);
        __syncthreads();   // previous tile fully consumed (and the mbarrier initialised)
        if (a.x0 == nullptr) {
            // fused feature assembly (gad_deform_fwd_ell with raw inputs): x_comp | f | uu staged by TMA
            // into the not-yet-used Xn buffer (dim + 2 <= CE floats per node), rows assembled into Xc
            const uint32_t xc_bytes = (uint32_t)NT * (uint32_t)a.dim * 4u, sc_bytes = (uint32_t)NT * 4u;
            const float* xc_g = a.x_comp + (size_t)n0 * a.dim;
            const float* f_g = a.f ? a.f + n0 : nullptr;
            const float* uu_g = a.uu ? a.uu + n0 : nullptr;
            const bool stage = (NT % 4 == 0) && ((reinterpret_cast<uintptr_t>(xc_g) | reinterpret_cast<uintptr_t>(f_g) |
                                                   reinterpret_cast<uintptr_t>(uu_g)) & 15) == 0 &&
                               (xc_bytes % 16 == 0);
            unsigned char* st_xc = Xn;
            unsigned char* st_f = st_xc + xc_bytes;
            unsigned char* st_uu = st_f + (a.f ? sc_bytes : 0u);
            const uint32_t tx = (ELLS ? (uint32_t)NT * 16u : 0u) +
                                (stage ? xc_bytes + (a.f ? sc_bytes : 0u) + (a.uu ? sc_bytes : 0u) : 0u);
            if (tid == 0 && tx) {
                fence_proxy_async_smem();
                mbar_expect_tx(bar, tx);
                if (ELLS) bulk_g2s(smem + lay.ein, a.ell_in + e0, (uint32_t)NT * 16u, bar);
                if (stage) {
                    bulk_g2s(st_xc, xc_g, xc_bytes, bar);
                    if (a.f) bulk_g2s(st_f, f_g, sc_bytes, bar);
                    if (a.uu) bulk_g2s(st_uu, uu_g, sc_bytes, bar);
                }
            }
            load_mu<CE>(a, Mu, 0, tile);
            if (tx) {
                mbar_wait(bar, parity);
                parity ^= 1;
            }
            assemble_rows<CE>(a, n0, NT, stage, st_xc, st_f, st_uu, Xc, a.states);
        } else {
        const float* x0t = a.x0 + (size_t)n0 * CE;
        const bool bulk_x = ((reinterpret_cast<uintptr_t>(x0t) & 15) == 0) && (((uint32_t)NT * RB) % 16 == 0);
        const uint32_t tx = (ELLS ? (uint32_t)NT * 16u : 0u) + (bulk_x ? (uint32_t)NT * RB : 0u);
        if (tid == 0 && tx) {
            fence_proxy_async_smem();
            mbar_expect_tx(bar, tx);
            if (ELLS) bulk_g2s(smem + lay.ein, a.ell_in + e0, (uint32_t)NT * 16u, bar);
            if (bulk_x) bulk_g2s(Xc, x0t, (uint32_t)NT * RB, bar);
        }
        if (!bulk_x)
            for (int i = tid; i < NT; i += nthr) sts_row<CE>(Xc, i * RB, load_row<CE>(a.x0, (int64_t)n0 + i));
        load_mu<CE>(a, Mu, 0, tile);
        if (tx) {
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        }
        __syncthreads();
        EllView<ELLS> Ein{ELLS ? reinterpret_cast<const uint4*>(smem + lay.ein) : a.ell_in + e0};

        for (int l = 0; l < a.L; ++l) {
            if (a.Lw > 1 && l > 0) {
                load_mu<CE>(a, Mu, l, tile);
                __syncthreads();
            }
            const float h = a.tau[l];
            const bool last = (l == a.L - 1);
            float* st_out = (a.states && !last) ? a.states + (size_t)(l + 1) * state_stride : nullptr;
            if constexpr (METHOD == GAD_METHOD_EULER) {
                float Mr[MUSZ];   // (M, u) in registers for the whole layer: no broadcast loads per node
#pragma unroll
                for (int t = 0; t < MUSZ; ++t) Mr[t] = Mu[t];
                uint4 e_nx = (tid < NT) ? Ein.get(tid) : make_uint4(0, 0, 0, 0);
                for (int i = tid; i < NT; i += nthr) {
                    const uint4 e = e_nx;
                    if (i + nthr < NT) e_nx = Ein.get(i + nthr);
                    const Row<CE> y = lds_row<CE>(Xc, i * RB);
                    const Row<CE> k = ell_feval<CE, W>(Xc, e, y, Mr);
                    Row<CE> xn;
#pragma unroll
                    for (int c = 0; c < CE; ++c) xn.v[c] = fmaf(h, k.v[c], y.v[c]);
                    sts_row<CE>(Xn, i * RB, xn);
                    if (st_out) store_row<CE>(st_out, (int64_t)n0 + i, xn);
                    if (last) store_dims<CE>(a.x_phys, (int64_t)n0 + i, a.dim, xn);   // decoder = identity slice
                }
                __syncthreads();
                unsigned char* t = Xc;
                Xc = Xn;
                Xn = t;
            } else {
                // classical RK4 on F(y) = A(y) y - y (extension, SURVEY A.1): the stage input lives in
                // the ping-pong buffers, the step's base state and the k-accumulator in XB / AC.
                const float cin[4] = {0.5f * h, 0.5f * h, h, 0.f};
                const float wacc[4] = {1.f, 2.f, 2.f, 1.f};
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    for (int i = tid; i < NT; i += nthr) {
                        const uint4 e = Ein.get(i);
                        const Row<CE> y = lds_row<CE>(Xc, i * RB);
                        const Row<CE> k = ell_feval<CE, W>(Xc, e, y, Mu);
                        Row<CE> base, acc, out;
                        if (s == 0) {
                            base = y;
                            acc = k;
                            sts_row<CE>(XB, i * RB, y);
                        } else {
                            base = lds_row<CE>(XB, i * RB);
                            acc = lds_row<CE>(AC, i * RB);
#pragma unroll
                            for (int c = 0; c < CE; ++c) acc.v[c] = fmaf(wacc[s], k.v[c], acc.v[c]);
                        }
                        if (s < 3) {
                            sts_row<CE>(AC, i * RB, acc);
#pragma unroll
                            for (int c = 0; c < CE; ++c) out.v[c] = fmaf(cin[s], k.v[c], base.v[c]);
                        } else {
#pragma unroll
                            for (int c = 0; c < CE; ++c) out.v[c] = fmaf(h * (1.0f / 6.0f), acc.v[c], base.v[c]);
                            if (st_out) store_row<CE>(st_out, (int64_t)n0 + i, out);
                            if (last) store_dims<CE>(a.x_phys, (int64_t)n0 + i, a.dim, out);
                        }
                        sts_row<CE>(Xn, i * RB, out);
                    }
                    __syncthreads();
                    unsigned char* t = Xc;
                    Xc = Xn;
                    Xn = t;
                }
            }
        }
    }
}

// ============================================================================================
// backward of one tile (shared by the backward and the train kernels)
// ============================================================================================
// On entry (all visible to the CTA): X = x^{L-1} rows, GS = dL/dx^L rows, Mu = weights of layer
// L-1.  acc: per-thread (G_M, G_u[, g_tau]) accumulators, zero on entry.
// FUSED_LAST (k_ell_train): the caller has already run phase A of layer L-1 inside its last forward
// layer (ell_feval_bwd_dst) and synchronised the CTA: GO / P / DL / GS hold that pass's rows, and
// acc_in / gtau_in its accumulators; the loop starts at phase B of layer L-1.  Then phase A also skips
// what nothing reads: g_tau terms without a g_tau column, and M t and the row stores of a layer that
// is followed by no source pass.
template <int CE, int W, bool ELLS, bool FUSED_LAST = false>
__device__ __forceinline__ void tile_backward(const Args& a, int tile, int n0, int NT, unsigned char* X,
                                              unsigned char* GO, unsigned char* P, unsigned char* DL,
                                              unsigned char* GS, const EllView<ELLS>& Ein,
                                              const EllView<ELLS>& Eout, float* Mu, float* red,
                                              const float* acc_in = nullptr, float gtau_in = 0.f) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    constexpr int NACC = MUSZ + 1;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const bool per_layer = (a.Lw > 1);
    const int slots = per_layer ? a.L : 1;
    const size_t state_stride = (size_t)a.N * CE;
    const bool need_gtau = !FUSED_LAST || per_layer || a.tau_partials != nullptr;
    float acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) acc[k] = FUSED_LAST ? acc_in[k] : 0.f;

    for (int l = a.L - 1; l >= 0; --l) {
        if (per_layer && l < a.L - 1) {
            load_mu<CE>(a, Mu, l, tile);
            __syncthreads();
        }
        const float b = a.tau[l];
        const bool fused = FUSED_LAST && l == a.L - 1;
        float gtau = fused ? gtau_in : 0.f;
        // ---- phase A: destination pass ------------------------------------------------------
        if (!fused) {
            const bool store = !FUSED_LAST || (l > 0) || (a.g_x0 != nullptr);   // a source pass reads the rows
            uint4 e_nx = (tid < NT) ? Ein.get(tid) : make_uint4(0, 0, 0, 0);
            for (int i = tid; i < NT; i += nthr) {
                const uint4 e = e_nx;
                if (i + nthr < NT) e_nx = Ein.get(i + nthr);
                const Row<CE> xi = lds_row<CE>(X, i * RB);
                const Row<CE> gp = lds_row<CE>(GS, i * RB);
                Row<CE> go;
#pragma unroll
                for (int c = 0; c < CE; ++c) go.v[c] = b * gp.v[c];
                Row<CE> p, t, o;
                float D, lse;
                ell_bwd_dst<CE, W>(X, e, xi, go, Mu, p, D, lse, t, o);
                if (need_gtau) {
#pragma unroll
                    for (int c = 0; c < CE; ++c) gtau = fmaf(gp.v[c], o.v[c] - xi.v[c], gtau);
                }
#pragma unroll
                for (int aa = 0; aa < CE; ++aa)
#pragma unroll
                    for (int bb = 0; bb < CE; ++bb) acc[aa * CE + bb] = fmaf(xi.v[aa], t.v[bb], acc[aa * CE + bb]);
#pragma unroll
                for (int bb = 0; bb < CE; ++bb) acc[CE * CE + bb] += t.v[bb];
                if (store) {
                    const Row<CE> Mt = apply_M<CE>(Mu, t);
                    Row<CE> gs;
#pragma unroll
                    for (int c = 0; c < CE; ++c) gs.v[c] = fmaf(1.0f - b, gp.v[c], Mt.v[c]);   // Euler: a = 1
                    sts_row<CE>(P, i * RB, p);
                    *reinterpret_cast<float2*>(DL + (size_t)i * 8) = make_float2(D, lse);
                    sts_row<CE>(GO, i * RB, go);
                    sts_row<CE>(GS, i * RB, gs);
                }
            }
        }
        const bool need_src = (l > 0) || (a.g_x0 != nullptr);
        if (need_src) {
            if (!fused) __syncthreads();   // P, DL, GO visible; every gather of X done
            // ---- phase B: source pass -------------------------------------------------------
            const float* xprev_g = (l > 0) ? a.states + (size_t)(l - 1) * state_stride : nullptr;
            uint4 e_nx = (tid < NT) ? Eout.get(tid) : make_uint4(0, 0, 0, 0);
            for (int j = tid; j < NT; j += nthr) {
                const uint4 e = e_nx;
                if (j + nthr < NT) e_nx = Eout.get(j + nthr);
                Row<CE> xprev;
                if (xprev_g) xprev = load_row_cg<CE>(xprev_g, (int64_t)n0 + j);   // issued early, used last
                const Row<CE> xj = lds_row<CE>(X, j * RB);
                const Row<CE> sc = ell_bwd_src<CE, W>(P, GO, DL, e, xj);
                Row<CE> g = lds_row<CE>(GS, j * RB);
#pragma unroll
                for (int c = 0; c < CE; ++c) g.v[c] += sc.v[c];
                sts_row<CE>(GS, j * RB, g);
                if (xprev_g) sts_row<CE>(X, j * RB, xprev);
                else if (a.g_x0) store_row<CE>(a.g_x0, (int64_t)n0 + j, g);
            }
            __syncthreads();   // GS / X of the next layer visible; gathers of P / DL / GO done
        }
        if (per_layer) {
            acc[NACC - 1] = gtau;
            block_reduce<NACC>(acc, red, a.partials + ((size_t)tile * slots + l) * NACC);
#pragma unroll
            for (int k = 0; k < NACC; ++k) acc[k] = 0.f;
        } else if (a.tau_partials) {
            float one[1] = {gtau};
            block_reduce<1>(one, red, a.tau_partials + (size_t)tile * a.L + l);
        }
    }
    if (!per_layer) block_reduce<NACC>(acc, red, a.partials + (size_t)tile * NACC);
}

template <int CE, int W, bool ELLS>
__global__ void __launch_bounds__(GAD_ELL_MAXT, GAD_ELL_MINB) k_ell_bwd(const Args a) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const Layout lay = make_layout(CE, KIND_BWD, a.cap_nodes, ELLS, (nthr + 31) >> 5);
    unsigned char* X = smem + lay.xa;
    unsigned char* GO = smem + lay.xb;
    unsigned char* P = smem + lay.p;
    unsigned char* GS = smem + lay.gs;
    unsigned char* DL = smem + lay.dl;
    float* Mu = reinterpret_cast<float*>(smem + lay.mu);
    float* red = reinterpret_cast<float*>(smem + lay.red);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + lay.bar);
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    uint32_t parity = 0;
    const size_t state_stride = (size_t)a.N * CE;

    for (int tile = blockIdx.x; tile < a.T; tile += gridDim.x) {
        int n0, NT, e0;
        tile_range(a, tile, n0, NT, e0);
        __syncthreads();
        const float* xl = a.states + (size_t)(a.L - 1) * state_stride + (size_t)n0 * CE;
        const bool bulk_x = ((reinterpret_cast<uintptr_t>(xl) & 15) == 0) && (((uint32_t)NT * RB) % 16 == 0);
        const uint32_t tx = (ELLS ? 2u * (uint32_t)NT * 16u : 0u) + (bulk_x ? (uint32_t)NT * RB : 0u);
        if (tid == 0 && tx) {
            fence_proxy_async_smem();
            mbar_expect_tx(bar, tx);
            if (ELLS) {
                bulk_g2s(smem + lay.ein, a.ell_in + e0, (uint32_t)NT * 16u, bar);
                bulk_g2s(smem + lay.eout, a.ell_out + e0, (uint32_t)NT * 16u, bar);
            }
            if (bulk_x) bulk_g2s(X, xl, (uint32_t)NT * RB, bar);
        }
        if (!bulk_x)
            for (int i = tid; i < NT; i += nthr) sts_row<CE>(X, i * RB, load_row_cg<CE>(xl, i));
        // cotangent of x_phys = x^L[:, :dim]  ->  dL/dx^L (zero in the other channels)
        for (int i = tid; i < NT; i += nthr) sts_row<CE>(GS, i * RB, load_dims<CE>(a.g_xphys, (int64_t)n0 + i, a.dim));
        const int lw = (a.Lw > 1) ? a.L - 1 : 0;
        load_mu<CE>(a, Mu, lw, tile);
        if (tx) {
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        __syncthreads();
        EllView<ELLS> Ein{ELLS ? reinterpret_cast<const uint4*>(smem + lay.ein) : a.ell_in + e0};
        EllView<ELLS> Eout{ELLS ? reinterpret_cast<const uint4*>(smem + lay.eout) : a.ell_out + e0};
        tile_backward<CE, W, ELLS>(a, tile, n0, NT, X, GO, P, DL, GS, Ein, Eout, Mu, red);
    }
}

// ============================================================================================
// backward of one tile through classical RK4 steps (the forward of k_ell_fwd<..., GAD_METHOD_RK4>)
// ============================================================================================
// One step  y' = y + h/6 (k1 + 2 k2 + 2 k3 + k4),  k_s = F(y_s),  y_1 = y, y_2 = y + h/2 k1, y_3 = y + h/2 k2,
// y_4 = y + h k3,  F(y) = A(y) y - y.  With g = dL/dy' and  vjp(x, c) = J_F(x)^T c = (d(A x)/dx)^T c - c :
//     c4 = h/6 g              a4 = vjp(y4, c4)
//     c3 = h/3 g + h   a4     a3 = vjp(y3, c3)
//     c2 = h/3 g + h/2 a3     a2 = vjp(y2, c2)
//     c1 = h/6 g + h/2 a2     a1 = vjp(y1, c1)          dL/dy = g + a1 + a2 + a3 + a4
// Only the step inputs y = x^l are saved by the forward (states[l]); the stage inputs are recomputed (three
// F-evaluations, same arithmetic as the forward).  Every vjp is the destination / source pass pair of the Euler
// backward with b = 1, and adds its (G_M, G_u) terms to the same per-thread accumulators.  Buffers (rows of CE
// floats per node): Y, Y2, Y3, Y4, G (step cotangent), AB (g + sum a_s), C (current cotangent / vjp result), GO, P.
template <int CE, int W, bool ELLS>
__device__ __forceinline__ void tile_backward_rk4(const Args& a, int tile, int n0, int NT, unsigned char* smem,
                                                  const Layout& lay, const EllView<ELLS>& Ein,
                                                  const EllView<ELLS>& Eout, float* Mu, float* red) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    constexpr int NACC = MUSZ + 1;
    const int tid = threadIdx.x, nthr = blockDim.x;
    unsigned char* Y = smem + lay.xa;
    unsigned char* GO = smem + lay.xb;
    unsigned char* P = smem + lay.p;
    unsigned char* C = smem + lay.gs;
    unsigned char* DL = smem + lay.dl;
    unsigned char* Y2 = smem + lay.y2;
    unsigned char* Y3 = smem + lay.y3;
    unsigned char* Y4 = smem + lay.y4;
    unsigned char* G = smem + lay.g;
    unsigned char* AB = smem + lay.ab;
    const bool per_layer = (a.Lw > 1);
    const int slots = per_layer ? a.L : 1;
    const size_t state_stride = (size_t)a.N * CE;
    float acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) acc[k] = 0.f;

    for (int l = a.L - 1; l >= 0; --l) {
        if (per_layer) {
            __syncthreads();
            load_mu<CE>(a, Mu, l, tile);
        }
        const float h = a.tau[l];
        const float h6 = h * (1.0f / 6.0f), h3 = 2.0f * h6, h2 = 0.5f * h;
        const float* yl = a.states + (size_t)l * state_stride;
        for (int i = tid; i < NT; i += nthr) sts_row<CE>(Y, i * RB, load_row_cg<CE>(yl, (int64_t)n0 + i));
        __syncthreads();
        // ---- stage inputs y2, y3, y4 (the forward's arithmetic)
#pragma unroll 1
        for (int sidx = 0; sidx < 3; ++sidx) {
            const unsigned char* src = (sidx == 0) ? Y : ((sidx == 1) ? Y2 : Y3);
            unsigned char* dst = (sidx == 0) ? Y2 : ((sidx == 1) ? Y3 : Y4);
            const float cs = (sidx == 2) ? h : h2;
            for (int i = tid; i < NT; i += nthr) {
                const uint4 e = Ein.get(i);
                const Row<CE> y = lds_row<CE>(src, i * RB);
                const Row<CE> k = ell_feval<CE, W>(src, e, y, Mu);
                const Row<CE> base = lds_row<CE>(Y, i * RB);
                Row<CE> out;
#pragma unroll
                for (int c = 0; c < CE; ++c) out.v[c] = fmaf(cs, k.v[c], base.v[c]);
                sts_row<CE>(dst, i * RB, out);
            }
            __syncthreads();
        }
        // ---- four cotangent passes, stage 4 first
#pragma unroll 1
        for (int ps = 0; ps < 4; ++ps) {
            const unsigned char* Xs = (ps == 0) ? Y4 : ((ps == 1) ? Y3 : ((ps == 2) ? Y2 : Y));
            for (int i = tid; i < NT; i += nthr) {          // destination pass, b = 1
                const uint4 e = Ein.get(i);
                const Row<CE> xi = lds_row<CE>(Xs, i * RB);
                Row<CE> c;
                if (ps == 0) {
                    const Row<CE> g = lds_row<CE>(G, i * RB);
#pragma unroll
                    for (int ch = 0; ch < CE; ++ch) c.v[ch] = h6 * g.v[ch];
                } else {
                    c = lds_row<CE>(C, i * RB);
                }
                Row<CE> p, t, o;
                float D, lse;
                ell_bwd_dst<CE, W>(Xs, e, xi, c, Mu, p, D, lse, t, o);
#pragma unroll
                for (int aa = 0; aa < CE; ++aa)
#pragma unroll
                    for (int bb = 0; bb < CE; ++bb) acc[aa * CE + bb] = fmaf(xi.v[aa], t.v[bb], acc[aa * CE + bb]);
#pragma unroll
                for (int bb = 0; bb < CE; ++bb) acc[CE * CE + bb] += t.v[bb];
                const Row<CE> Mt = apply_M<CE>(Mu, t);
                sts_row<CE>(P, i * RB, p);
                *reinterpret_cast<float2*>(DL + (size_t)i * 8) = make_float2(D, lse);
                sts_row<CE>(GO, i * RB, c);
                sts_row<CE>(C, i * RB, Mt);
            }
            __syncthreads();
            const float wg = (ps == 2) ? h6 : h3, wa = (ps == 0) ? h : h2;     // next cotangent = wg g + wa a_s
            for (int j = tid; j < NT; j += nthr) {          // source pass + node-local bookkeeping
                const uint4 e = Eout.get(j);
                const Row<CE> xj = lds_row<CE>(Xs, j * RB);
                const Row<CE> sc = ell_bwd_src<CE, W>(P, GO, DL, e, xj);
                const Row<CE> r = lds_row<CE>(C, j * RB);
                const Row<CE> cj = lds_row<CE>(GO, j * RB);
                const Row<CE> g = lds_row<CE>(G, j * RB);
                Row<CE> as, ab;
#pragma unroll
                for (int ch = 0; ch < CE; ++ch) as.v[ch] = (r.v[ch] + sc.v[ch]) - cj.v[ch];
                if (ps == 0) {
#pragma unroll
                    for (int ch = 0; ch < CE; ++ch) ab.v[ch] = g.v[ch] + as.v[ch];
                } else {
                    ab = lds_row<CE>(AB, j * RB);
#pragma unroll
                    for (int ch = 0; ch < CE; ++ch) ab.v[ch] += as.v[ch];
                }
                if (ps < 3) {
                    Row<CE> cn;
#pragma unroll
                    for (int ch = 0; ch < CE; ++ch) cn.v[ch] = fmaf(wg, g.v[ch], wa * as.v[ch]);
                    sts_row<CE>(AB, j * RB, ab);
                    sts_row<CE>(C, j * RB, cn);
                } else {
                    sts_row<CE>(G, j * RB, ab);             // dL/dx^l: the cotangent of the previous step
                    if (l == 0 && a.g_x0) store_row<CE>(a.g_x0, (int64_t)n0 + j, ab);
                }
            }
            __syncthreads();
        }
        if (per_layer) {
            acc[NACC - 1] = 0.f;
            block_reduce<NACC>(acc, red, a.partials + ((size_t)tile * slots + l) * NACC);
#pragma unroll
            for (int k = 0; k < NACC; ++k) acc[k] = 0.f;
        }
    }
    if (!per_layer) block_reduce<NACC>(acc, red, a.partials + (size_t)tile * NACC);
}

template <int CE, int W, bool ELLS>
__global__ void __launch_bounds__(GAD_ELL_MAXT, GAD_ELL_MINB) k_ell_bwd_rk4(const Args a) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const Layout lay = make_layout(CE, KIND_BWD_RK4, a.cap_nodes, ELLS, (nthr + 31) >> 5);
    unsigned char* G = smem + lay.g;
    float* Mu = reinterpret_cast<float*>(smem + lay.mu);
    float* red = reinterpret_cast<float*>(smem + lay.red);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + lay.bar);
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    uint32_t parity = 0;
    for (int tile = blockIdx.x; tile < a.T; tile += gridDim.x) {
        int n0, NT, e0;
        tile_range(a, tile, n0, NT, e0);
        __syncthreads();
        const uint32_t tx = ELLS ? 2u * (uint32_t)NT * 16u : 0u;
        if (tid == 0 && tx) {
            fence_proxy_async_smem();
            mbar_expect_tx(bar, tx);
            bulk_g2s(smem + lay.ein, a.ell_in + e0, (uint32_t)NT * 16u, bar);
            bulk_g2s(smem + lay.eout, a.ell_out + e0, (uint32_t)NT * 16u, bar);
        }
        // cotangent of x_phys = x^L[:, :dim]  ->  dL/dx^L (zero in the other channels)
        for (int i = tid; i < NT; i += nthr) sts_row<CE>(G, i * RB, load_dims<CE>(a.g_xphys, (int64_t)n0 + i, a.dim));
        const int lw = (a.Lw > 1) ? a.L - 1 : 0;
        load_mu<CE>(a, Mu, lw, tile);
        if (tx) {
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        __syncthreads();
        EllView<ELLS> Ein{ELLS ? reinterpret_cast<const uint4*>(smem + lay.ein) : a.ell_in + e0};
        EllView<ELLS> Eout{ELLS ? reinterpret_cast<const uint4*>(smem + lay.eout) : a.ell_out + e0};
        tile_backward_rk4<CE, W, ELLS>(a, tile, n0, NT, smem, lay, Ein, Eout, Mu, red);
    }
}

// Programmatic dependent launch (sm_90+): `launch_dependents` lets the NEXT kernel of the stream start
// its CTAs while this one still runs; `wait` blocks until every prerequisite grid has completed and
// its memory is visible.  Both are no-ops when the launch carries no programmatic dependency.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ============================================================================================
// tail of the training step: reduction of the per-tile partials, chain rule, Adam, refold
// ============================================================================================
// Run by ONE CTA per launch.  What it costs is the length of its dependent instruction stream
// (every stage is a few hundred mostly-serial instructions of one warp), not bandwidth, so it is
// split in two:
//   tail_prepare  everything that does not depend on this step's partials -- shared-memory mirrors
//                 of the flat parameter / gradient vectors (cp.async), the Adam moments of the
//                 thread's parameter in registers, the structurally-zero gradient entries;
//   tail_finish   partials -> fixed-order fp64 column sums -> chain rule to the Linear parameters
//                 (src/GRAND_plus.py:225-226 folded, tail_math.cuh) -> Adam (src/run_GNN.py:88,128,131)
//                 on the mirror -> refold of (M, u) for the next launch, all through shared memory
//                 with 32-bit offsets: one L2 round trip (the partials) and four barriers.
// When the whole grid is resident at once the training kernel adds a reducer CTA that owns no tile:
// it runs tail_prepare while the tiles are being processed, waits until every tile CTA has checked
// in, and runs tail_finish.  Otherwise the last tile CTA to finish runs both parts.  The host checks
// plan_tail().ok (and that Wq / bq / Wk, gWq / gbq / gWk / gbk are views of params / grads) and
// otherwise launches with tail = 0 followed by the stand-alone kernels.
struct TailPlan {
    uint32_t colsum, wp, gmu, ps, gs, stage;   // byte offsets into the scratch
    int ncol, ntau, nloss, ncolT, TC;          // columns of the three partial arrays; tiles per chunk
    int nps;                                   // floats mirrored in `ps`
    uint32_t stage_bytes;                      // room behind `stage` (partials chunks; received peer gradients)
    bool ok;
};

__host__ __device__ inline TailPlan plan_tail(int CE, int Lw, int L, int C, bool tau_cols, bool loss_col,
                                              long long n_params, int T, int nwarps, size_t scratch_bytes) {
    const int MUSZ = CE * CE + CE, NACC = MUSZ + 1;
    TailPlan p{};
    p.ncol = (Lw > 1 ? L : 1) * NACC;
    p.ntau = tau_cols ? L : 0;
    p.nloss = loss_col ? 1 : 0;
    p.ncolT = p.ncol + p.ntau + p.nloss;
    // Adam (n_params > 0): mirror of the whole flat vector; else [Wq | bq | Wk]
    const long long nps = n_params > 0 ? n_params : (long long)Lw * (2 * C * C + C);
    size_t o = 0;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o = (o + bytes + 15) & ~size_t(15);
        return (uint32_t)at;
    };
    p.colsum = take((size_t)p.ncolT * sizeof(double));
    p.wp = take((size_t)p.ncolT * nwarps * sizeof(double));
    p.gmu = take((size_t)Lw * MUSZ * sizeof(float));
    p.ps = take((size_t)nps * sizeof(float));
    p.gs = take((size_t)n_params * sizeof(float));
    p.stage = (uint32_t)o;
    p.nps = (int)nps;
    p.ok = nps < (1 << 24) && o + (size_t)p.ncolT * sizeof(float) <= scratch_bytes;
    if (!p.ok) return p;
    p.stage_bytes = (uint32_t)(scratch_bytes - o);
    long long tc = (long long)((scratch_bytes - o) / sizeof(float)) / p.ncolT;
    if (tc > T) tc = T;
    if (tc > 32) tc &= ~31LL;
    p.TC = (int)tc;
    return p;
}

struct TailCtx {
    TailPlan tp;
    uint32_t oWq, obq, oWk;        // float offsets of the weights in the `ps` mirror
    uint32_t ogWq, ogbq, ogWk;     // float offsets of their gradients in the `gs` mirror (Adam)
    float m0, v0;                  // Adam moments of parameter `tid`
    uint32_t seq;                  // sequence number of this launch's peer exchange (world > 1)
};

// ---- gradient all-reduce over peer memory, inside the tail ----------------------------------------
// Every rank stores { value, seq } words (8 bytes: single-copy atomic, so the tag travels with the
// data and no fence is needed -- the LL protocol of NCCL) into slot [seq & 1][rank] of EVERY
// rank's receive buffer, then sums slots [seq & 1][0 .. world) of its own buffer in rank order
// once their tags match.  Same order on every rank: the reduced gradient, hence the parameters,
// stay bit-identical across ranks.  Two parities make the buffers safe to reuse: a peer can only
// overwrite parity p two exchanges later, which needs this rank's contribution to the exchange
// in between, which this rank sends only after it has finished reading parity p.
__device__ __forceinline__ void st_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Every (destination rank, parameter) word has its own thread for the store and every (source rank,
// parameter) word its own thread for the poll, so the `world` NVLink round trips of a parameter are in
// flight together instead of one after the other; the received values go through shared memory (V,
// [world][n]) and are summed in RANK ORDER by one thread per parameter -- same bits on every rank.
// The wait is bounded: a peer that died, skipped a step or took another route (NCCL) leaves its tag
// stale; after `timeout_ns` the CTA gives up, returns false and the caller raises the device error
// word instead of taking the Adam step (the host checks it: DeformerTrainer.check_peer).
__device__ __forceinline__ bool peer_allreduce(const Args& a, float* Gs, float* V, int n, uint32_t seq,
                                               unsigned long long* const* s_peers, volatile int* s_fail) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    const size_t slot = (size_t)(seq & 1u) * a.world;
    const int total = a.world * n;
#pragma unroll 1
    for (int idx = tid; idx < total; idx += nthr) {
        const int r = idx / n, i = idx - r * n;
        const unsigned long long word = ((unsigned long long)seq << 32) | (unsigned long long)__float_as_uint(Gs[i]);
        st_sys_u64(s_peers[r] + (slot + a.rank) * n + i, word);
    }
    const unsigned long long* own = s_peers[a.rank] + slot * n;   // [world][n] words of this parity, contiguous
    const unsigned long long t0 = globaltimer_ns();
    // polls: four words per thread in flight at a time (a sys-scope load is a full L2 round trip; polling a
    // thread's words one after the other would put world * n / nthr of them in series)
#pragma unroll 1
    for (int base = 0; base < total; base += 4 * nthr) {
        int idx[4];
        bool need[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            idx[k] = base + k * nthr + tid;
            need[k] = idx[k] < total;
        }
        uint32_t spins = 0;
        while (need[0] || need[1] || need[2] || need[3]) {
            unsigned long long w[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (need[k]) w[k] = ld_sys_u64(own + idx[k]);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (need[k] && (uint32_t)(w[k] >> 32) == seq) {
                    V[idx[k]] = __uint_as_float((uint32_t)w[k]);
                    need[k] = false;
                }
            if ((++spins & 63u) == 0u) {
                if (*s_fail) break;
                if (globaltimer_ns() - t0 > a.peer_timeout_ns) {
                    *s_fail = 1;
                    break;
                }
            }
        }
    }
    __syncthreads();
    if (*s_fail) return false;
    float* grads_out = const_cast<float*>(a.grads);
#pragma unroll 1
    for (int i = tid; i < n; i += nthr) {
        float sum = 0.f;
#pragma unroll 1
        for (int r = 0; r < a.world; ++r) sum += V[r * n + i];
        Gs[i] = sum;
        grads_out[i] = sum;
    }
    return true;
}

template <int CE>
__device__ __forceinline__ void tail_prepare(const Args& a, unsigned char* scratch, uint32_t scratch_bytes, TailCtx& cx) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    const bool adam = a.tail >= 2;
    const int np = adam ? (int)a.n_params : 0;
    const int C = a.C, rows = a.Lw * C;
    cx.tp = plan_tail(CE, a.Lw, a.L, C, a.tau_partials && a.g_tau, a.loss_partials && a.loss, np, a.T,
                      (nthr + 31) >> 5, scratch_bytes);
    float* Ps = reinterpret_cast<float*>(scratch + cx.tp.ps);
    float* Gs = reinterpret_cast<float*>(scratch + cx.tp.gs);
    double* colsum = reinterpret_cast<double*>(scratch + cx.tp.colsum);
    cx.m0 = cx.v0 = 0.f;
    cx.seq = (adam && a.world > 1 && a.peers) ? __ldcg(a.peer_seq) + 1u : 0u;
    if (adam) {
        cx.oWq = (uint32_t)(a.Wq - a.params);
        cx.obq = (uint32_t)(a.bq - a.params);
        cx.oWk = (uint32_t)(a.Wk - a.params);
        cx.ogWq = (uint32_t)(a.gWq - a.grads);
        cx.ogbq = (uint32_t)(a.gbq - a.grads);
        cx.ogWk = (uint32_t)(a.gWk - a.grads);
        if (tid < np) {
            cx.m0 = __ldcg(a.exp_avg + tid);
            cx.v0 = __ldcg(a.exp_avg_sq + tid);
        }
        tail::stage_async(Ps, a.params, np);
        tail::stage_async(Gs, a.grads, np);   // entries the tail does not produce keep their value
    } else {
        cx.oWq = 0;
        cx.obq = (uint32_t)(rows * C);
        cx.oWk = cx.obq + (uint32_t)rows;
        cx.ogWq = cx.ogbq = cx.ogWk = 0;
        tail::stage_async(Ps + cx.oWq, a.Wq, rows * C);
        tail::stage_async(Ps + cx.obq, a.bq, rows);
        tail::stage_async(Ps + cx.oWk, a.Wk, rows * C);
    }
    for (int c = tid; c < cx.tp.ncolT; c += nthr) colsum[c] = 0.0;
    tail::stage_wait();
    __syncthreads();
    // structurally zero gradients: d/d lin_key.bias (softmax shift invariance) and the columns of
    // Wq / Wk that only ever multiply dead channels
    const int gbk_off = adam ? (int)(a.gbk - a.grads) : 0;
#pragma unroll 1
    for (int lo = tid; lo < rows; lo += nthr) {
        a.gbk[lo] = 0.0f;
        if (adam) Gs[gbk_off + lo] = 0.0f;
    }
    if (C > CE) {
        const int dead = C - CE;
#pragma unroll 1
        for (int idx = tid; idx < rows * dead; idx += nthr) {
            const int lo = idx / dead, o = lo * C + CE + (idx - lo * dead);
            a.gWq[o] = 0.0f;
            a.gWk[o] = 0.0f;
            if (adam) {
                Gs[cx.ogWq + o] = 0.0f;
                Gs[cx.ogWk + o] = 0.0f;
            }
        }
    }
}

template <int CE>
__device__ __forceinline__ void tail_finish(const Args& a, unsigned char* scratch, const TailCtx& cx,
                                            const tail::AdamCoef& coef, long long t_step, Tracer& tr) {
    constexpr int MUSZ = CE * CE + CE;
    constexpr int NACC = MUSZ + 1;
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = (nthr + 31) >> 5;
    const bool adam = a.tail >= 2;
    const int np = adam ? (int)a.n_params : 0;
    const int slots = a.Lw > 1 ? a.L : 1;
    const TailPlan& tp = cx.tp;
    const int ncol = tp.ncol, ntau = tp.ntau, nloss = tp.nloss, ncolT = tp.ncolT, TC = tp.TC;
    double* colsum = reinterpret_cast<double*>(scratch + tp.colsum);
    double* wp = reinterpret_cast<double*>(scratch + tp.wp);
    float* gMu_s = reinterpret_cast<float*>(scratch + tp.gmu);
    float* Ps = reinterpret_cast<float*>(scratch + tp.ps);
    float* Gs = reinterpret_cast<float*>(scratch + tp.gs);
    float* S = reinterpret_cast<float*>(scratch + tp.stage);

    // ---- (1) fixed-order column sums: lane = column, warp = contiguous range of tiles (two
    // interleaved fp64 chains), then the warps' sums in warp order; chunk by chunk
#pragma unroll 1
    for (int t0 = 0; t0 < a.T; t0 += TC) {
        const int nt = (a.T - t0 < TC) ? a.T - t0 : TC;
        float* S0 = S;
        float* S1 = S0 + nt * ncol;
        float* S2 = S1 + nt * ntau;
        tail::stage_async(S0, a.partials + (size_t)t0 * ncol, nt * ncol);
        if (ntau) tail::stage_async(S1, a.tau_partials + (size_t)t0 * a.L, nt * ntau);
        if (nloss) tail::stage_async(S2, a.loss_partials + t0, nt);
        tail::stage_wait();
        __syncthreads();
        const int tpw = (nt + nwarps - 1) / nwarps;
        const int tb = warp * tpw, te = (tb + tpw < nt) ? tb + tpw : nt;
#pragma unroll 1
        for (int c = lane; c < ncolT; c += 32) {
            const float* src = (c < ncol) ? S0 + c : ((c < ncol + ntau) ? S1 + (c - ncol) : S2);
            const int stride = (c < ncol) ? ncol : ((c < ncol + ntau) ? ntau : 1);
            double s0 = 0.0, s1 = 0.0;   // fp64: the per-tile partials cancel heavily across meshes
            int t = tb;
#pragma unroll 4
            for (; t + 1 < te; t += 2) {
                s0 += (double)src[t * stride];
                s1 += (double)src[(t + 1) * stride];
            }
            if (t < te) s0 += (double)src[t * stride];
            wp[warp * ncolT + c] = s0 + s1;
        }
        __syncthreads();
#pragma unroll 1
        for (int c = tid; c < ncolT; c += nthr) {
            double sd = colsum[c];
            for (int w = 0; w < nwarps; ++w) sd += wp[w * ncolT + c];
            colsum[c] = sd;
            if (t0 + TC >= a.T) {   // last chunk: the column is complete
                const float sv = (float)sd;
                if (c < ncol) {
                    const int l = c / NACC, k = c - l * NACC;
                    if (k < MUSZ) {
                        gMu_s[l * MUSZ + k] = sv;
                        a.gMu[l * MUSZ + k] = sv;
                    } else if (a.g_tau && slots > 1) {
                        a.g_tau[l] = sv;
                        if (adam) Gs[(a.g_tau - a.grads) + l] = sv;
                    }
                } else if (c < ncol + ntau) {
                    a.g_tau[c - ncol] = sv;
                    if (adam) Gs[(a.g_tau - a.grads) + (c - ncol)] = sv;
                } else {
                    a.loss[0] = sv * a.loss_scale;
                }
            }
        }
        __syncthreads();
    }
    tr.mark();   // partials reduced

    // ---- (2) chain rule: rows lo = l * C + o of Wq / Wk viewed as [Lw * C, C], live columns only
    // (same arithmetic, same order as tail::weight_grads); the bias rows go to the high threads
    const int C = a.C, rows = a.Lw * C;
    const int live = CE < C ? CE : C;
    const double cfold = a.cfold;
#pragma unroll 1
    for (int idx = tid; idx < rows * CE; idx += nthr) {
        const int aa = idx % CE, lo = idx / CE;
        if (aa >= live) continue;
        const int l = (a.Lw > 1) ? lo / C : 0;
        float dq, dk;
        tail::weight_grad_entry<CE>(Ps + cx.oWq + lo * C, Ps + cx.oWk + lo * C, Ps[cx.obq + lo], gMu_s + l * MUSZ, live, aa,
                                    cfold, dq, dk);
        const int o = lo * C + aa;
        a.gWq[o] = dq;
        a.gWk[o] = dk;
        if (adam) {
            Gs[cx.ogWq + o] = dq;
            Gs[cx.ogWk + o] = dk;
        }
    }
#pragma unroll 1
    for (int lo = nthr - 1 - tid; lo < rows; lo += nthr) {
        const int l = (a.Lw > 1) ? lo / C : 0;
        const float* wk = Ps + cx.oWk + lo * C;
        const float* Gu = gMu_s + l * MUSZ + CE * CE;
        double d = 0.0;
#pragma unroll
        for (int bb = 0; bb < CE; ++bb)
            if (bb < live) d += (double)wk[bb] * (double)Gu[bb];
        const float g = (float)(cfold * d);
        a.gbq[lo] = g;
        if (adam) Gs[cx.ogbq + lo] = g;
    }
    if (!adam) return;
    __syncthreads();
    if (cx.seq) {
        // data parallel: SUM all-reduce of the flat gradient over peer memory (NVLink), in place
        __shared__ unsigned long long* s_peers[GAD_MAX_PEERS];
        __shared__ int s_fail;
        if (tid < a.world) s_peers[tid] = reinterpret_cast<unsigned long long*>(a.peers[tid]);
        if (tid == 0) s_fail = (__ldcg(a.peer_seq + 1) != 0u) ? 1 : 0;   // an earlier exchange failed: do not wait again
        __syncthreads();
        const bool arrived = peer_allreduce(a, Gs, S, np, cx.seq, s_peers, &s_fail);   // S: the staging area is free now
        if (tid == 0) {
            *a.peer_seq = cx.seq;
            if (!arrived) a.peer_seq[1] = cx.seq;   // sticky error word: exchange `seq` timed out
        }
        __syncthreads();
        if (!arrived) return;                       // no Adam step, no refold: parameters keep their value
    }
    tr.mark();   // chain rule (+ gradient exchange)

    // ---- (3) Adam on the mirror ------------------------------------------------------------------
#pragma unroll 1
    for (int i = tid; i < np; i += nthr) {
        float m = cx.m0, v = cx.v0;
        if (i >= nthr) {
            m = __ldcg(a.exp_avg + i);
            v = __ldcg(a.exp_avg_sq + i);
        }
        const float pn = tail::adam_update(coef, Ps[i], Gs[i], m, v);
        Ps[i] = pn;
        a.params[i] = pn;
        a.exp_avg[i] = m;
        a.exp_avg_sq[i] = v;
    }
    if (tid == 0) a.step[0] = t_step;
    __syncthreads();
    tr.mark();   // Adam

    // ---- (4) refold (M, u) of the next step from the mirror ---------------------------------------
    tail::prepare_weights_t<CE>(Ps + cx.oWq, Ps + cx.obq, Ps + cx.oWk, a.Lw, C, cfold, a.Mu_next);
}

// ============================================================================================
// train: feature assembly + forward + mesh loss + backward of a tile, one launch
// ============================================================================================
// Replaces pack -> forward -> loss -> backward of the training step (src/run_GNN.py:99-131 with
// loss_type = mesh_loss): x_phys and its cotangent never leave the SM.  The layer states go to
// `states` (L2-resident scratch) on the way up and are read back by the same thread on the way
// down; ld.global.cg keeps those reads coherent.
// METHOD == GAD_METHOD_RK4: classical RK4 steps (the forward of k_ell_fwd<..., GAD_METHOD_RK4>, same
// expressions), the loss fused into stage 4 of the last step, then tile_backward_rk4.  The inputs are
// staged into the Y2 rows (untouched until the backward recomputes the stages) and the target into DL;
// the cotangent goes to the G rows, which tile_backward_rk4 reads as dL/dx^L.
// COT (loss_kind 2): the target rows hold a cotangent c of x_phys computed outside the model; the loss stage sets
// dL/dx^L = grad_scale * c and sums the pseudo-loss <x_phys, c>.  A template flag, so that the mesh-loss kernels
// compile to what they were before it existed.
template <int CE, int W, bool ELLS, int METHOD, bool COT = false>
__global__ void __launch_bounds__(GAD_ELL_MAXT, GAD_ELL_MINB) k_ell_train(const Args a) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const Layout lay = make_layout(CE, METHOD == GAD_METHOD_RK4 ? KIND_TRAIN_RK4 : KIND_BWD, a.cap_nodes, ELLS,
                                   (nthr + 31) >> 5);
    unsigned char* B0 = smem + lay.xa;
    unsigned char* B1 = smem + lay.xb;
    unsigned char* P = smem + lay.p;
    unsigned char* GS = smem + lay.gs;
    unsigned char* DL = smem + lay.dl;
    float* Mu = reinterpret_cast<float*>(smem + lay.mu);
    float* red = reinterpret_cast<float*>(smem + lay.red);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + lay.bar);
    __shared__ int s_last;
    __shared__ long long s_step;
    __shared__ tail::AdamCoef s_coef;
    // The next training step (same stream, programmatic dependency) may start its CTAs now: its
    // input staging below touches only data no kernel writes, so it overlaps this step's compute;
    // everything this step produces is consumed after pdl_wait().
    pdl_launch_dependents();
    Tracer tr{a.trace ? a.trace + (size_t)blockIdx.x * 64 : nullptr, 0};
    tr.mark();   // 0: kernel entry
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    uint32_t parity = 0;
    const size_t state_stride = (size_t)a.N * CE;
    // With a whole grid resident at once (T + 1 <= CTA slots) an EXTRA CTA, the last of the grid, is
    // the reducer: it owns no tile, prepares the tail while the tiles are processed, waits until every tile CTA
    // has checked in and then runs the tail.  Otherwise the last tile CTA to finish runs it.
    const int tile_ctas = a.tail_cta ? (int)gridDim.x - 1 : (int)gridDim.x;
    const bool reducer = a.tail_cta && (int)blockIdx.x == tile_ctas;

    for (int tile = reducer ? a.T : (int)blockIdx.x; tile < a.T; tile += tile_ctas) {
        int n0, NT, e0;
        tile_range(a, tile, n0, NT, e0);
        __syncthreads();
        // Inputs of the tile by 1-D TMA bulk copies: ELL rows to their buffers, x_comp | f | uu to a
        // staging area in the (not yet used) P buffer, the target mesh to the DL buffer.
        const uint32_t xc_bytes = (uint32_t)NT * (uint32_t)a.dim * 4u, sc_bytes = (uint32_t)NT * 4u;
        const float* xc_g = a.x_comp + (size_t)n0 * a.dim;
        const float* tg_g = a.target + (size_t)n0 * a.dim;
        const float* f_g = a.f ? a.f + n0 : nullptr;
        const float* uu_g = a.uu ? a.uu + n0 : nullptr;
        const bool stage = a.dim <= 2 && (NT % 4 == 0) &&
                           ((reinterpret_cast<uintptr_t>(xc_g) | reinterpret_cast<uintptr_t>(tg_g) |
                             reinterpret_cast<uintptr_t>(f_g) | reinterpret_cast<uintptr_t>(uu_g)) & 15) == 0;
        unsigned char* st_xc = (METHOD == GAD_METHOD_RK4) ? smem + lay.y2 : P;
        unsigned char* st_f = st_xc + xc_bytes;
        unsigned char* st_uu = st_f + (a.f ? sc_bytes : 0u);
        const uint32_t tx = (ELLS ? 2u * (uint32_t)NT * 16u : 0u) +
                            (stage ? 2u * xc_bytes + (a.f ? sc_bytes : 0u) + (a.uu ? sc_bytes : 0u) : 0u);
        if (tid == 0 && tx) {
            fence_proxy_async_smem();
            mbar_expect_tx(bar, tx);
            if (ELLS) {
                bulk_g2s(smem + lay.ein, a.ell_in + e0, (uint32_t)NT * 16u, bar);
                bulk_g2s(smem + lay.eout, a.ell_out + e0, (uint32_t)NT * 16u, bar);
            }
            if (stage) {
                bulk_g2s(st_xc, xc_g, xc_bytes, bar);
                if (a.f) bulk_g2s(st_f, f_g, sc_bytes, bar);
                if (a.uu) bulk_g2s(st_uu, uu_g, sc_bytes, bar);
                bulk_g2s(DL, tg_g, xc_bytes, bar);
            }
        }
        // Everything that only needs the step's INPUTS happens before the wait on the previous step, i.e.
        // in its shadow when the launches are chained by programmatic dependent launch.
        if (tx) {
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        tr.mark();   // 1: inputs landed
        // features = cat[x_comp, f, uu] + identity (zero-pad) encoder: src/GNN.py:225-239,75-83,270
        unsigned char* Xc = B0;
        unsigned char* Xn = B1;
        assemble_rows<CE>(a, n0, NT, stage, st_xc, st_f, st_uu, Xc, nullptr);   // x^0 reaches `states` from the first layer's loop, after the wait
        if (METHOD == GAD_METHOD_EULER && a.dim == 1 && stage) {
            // The Euler last layer overwrites the DL row of node i (8 bytes) with (D, lse) right after reading
            // node i's target.  A staged 1-D target is 4 bytes per node, so that row holds the targets of nodes
            // 2i and 2i+1, which other threads may not have read yet: move each target into its node's GS row
            // (unused until then) before the barrier.  At dim 2 the DL row of node i is node i's target.
            for (int i = tid; i < NT; i += nthr)
                reinterpret_cast<float*>(GS + i * RB)[0] = reinterpret_cast<const float*>(DL)[i];
        }
        __syncthreads();
        // previous step done (weights refolded, its reads of `states` finished): from here on this
        // step may read Mu / tau and write global memory
        pdl_wait();
        tr.mark();   // 2: predecessor done
        // Adam's bias corrections of THIS step (a serial fp64 chain) are worked out now by one thread
        // of every CTA, hidden behind the tile's work, so that whichever CTA runs the tail has them
        if (a.tail >= 2 && !a.tail_cta && tile == (int)blockIdx.x && tid == nthr - 1) {
            s_step = __ldcg(a.step) + 1;
            s_coef = tail::adam_coef(a.lr, a.beta1, a.beta2, a.eps, a.weight_decay, a.adam_grad_scale, s_step);
        }
        // (M, u): one L2 request per CTA (every thread loading it would hammer a single L2 line from
        // 2000 warps at once), then through shared memory
        for (int t = tid; t < MUSZ; t += nthr) Mu[t] = __ldcg(a.Mu + t);
        __syncthreads();
        EllView<ELLS> Ein{ELLS ? reinterpret_cast<const uint4*>(smem + lay.ein) : a.ell_in + e0};
        EllView<ELLS> Eout{ELLS ? reinterpret_cast<const uint4*>(smem + lay.eout) : a.ell_out + e0};

        if constexpr (METHOD == GAD_METHOD_EULER) {
        // ---- forward (Euler); the last layer also computes the loss, its cotangent and phase A
        // (destination pass) of the backward of that layer, from the same gathered rows
        for (int l = 0; l < a.L - 1; ++l) {
            if (a.Lw > 1 && l > 0) {
                for (int t = tid; t < MUSZ; t += nthr) Mu[t] = a.Mu[(size_t)l * MUSZ + t];
                __syncthreads();
            }
            const float h = __ldcg(a.tau + l);
            float* st_out = a.states + (size_t)(l + 1) * state_stride;
            float Mr[MUSZ];   // (M, u) in registers for the whole layer: no broadcast loads per node
#pragma unroll
            for (int t = 0; t < MUSZ; ++t) Mr[t] = Mu[t];
            uint4 e_nx = (tid < NT) ? Ein.get(tid) : make_uint4(0, 0, 0, 0);
            for (int i = tid; i < NT; i += nthr) {
                const uint4 e = e_nx;
                if (i + nthr < NT) e_nx = Ein.get(i + nthr);
                const Row<CE> y = lds_row<CE>(Xc, i * RB);
                if (l == 0) store_row<CE>(a.states, (int64_t)n0 + i, y);
                const Row<CE> k = ell_feval<CE, W>(Xc, e, y, Mr);
                Row<CE> xn;
#pragma unroll
                for (int c = 0; c < CE; ++c) xn.v[c] = fmaf(h, k.v[c], y.v[c]);
                sts_row<CE>(Xn, i * RB, xn);
                store_row<CE>(st_out, (int64_t)n0 + i, xn);
            }
            __syncthreads();
            tr.mark();   // 3 .. 2+L: forward layers
            unsigned char* t = Xc;
            Xc = Xn;
            Xn = t;
        }
        {
            // last layer, l = L-1: Xc = x^{L-1} (kept for the backward), Xn is free and takes the GO rows
            const int l = a.L - 1;
            if (a.Lw > 1 && l > 0) {
                for (int t = tid; t < MUSZ; t += nthr) Mu[t] = a.Mu[(size_t)l * MUSZ + t];
                __syncthreads();
            }
            const float h = __ldcg(a.tau + l);
            const bool src = (l > 0) || (a.g_x0 != nullptr);   // a source pass follows: the rows below are read
            const bool need_gtau = (a.Lw > 1) || (a.tau_partials != nullptr);
            const unsigned char* TG = (a.dim == 1) ? GS : DL;   // staged target of node i, see the feature assembly
            const uint32_t tg_rb = (a.dim == 1) ? RB : 8u;
            constexpr int NACC = MUSZ + 1;
            float acc[NACC];
#pragma unroll
            for (int k = 0; k < NACC; ++k) acc[k] = 0.f;
            float gtau = 0.f, loss_acc = 0.f;
            if (l == 0)   // L = 1: x^0 reaches `states` here
                for (int i = tid; i < NT; i += nthr) store_row<CE>(a.states, (int64_t)n0 + i, lds_row<CE>(Xc, i * RB));
            uint4 e_nx = (tid < NT) ? Ein.get(tid) : make_uint4(0, 0, 0, 0);
            for (int i = tid; i < NT; i += nthr) {
                const uint4 e = e_nx;
                if (i + nthr < NT) e_nx = Ein.get(i + nthr);
                const Row<CE> y = lds_row<CE>(Xc, i * RB);
                const int64_t gi = (int64_t)n0 + i;
                // x^L = y + h k -> x_phys, loss term and cotangent dL/dx^L of this node
                auto cot = [&](const Row<CE>& k) {
                    Row<CE> xn;
#pragma unroll
                    for (int c = 0; c < CE; ++c) xn.v[c] = fmaf(h, k.v[c], y.v[c]);
                    auto term = [&](float d) {   // adds d's loss term, returns its cotangent entry
                        if (a.loss_kind == 0) {
                            loss_acc += fabsf(d);
                            return (d > 0.f) ? a.grad_scale : ((d < 0.f) ? -a.grad_scale : 0.f);   // torch sign()
                        }
                        loss_acc = fmaf(d, d, loss_acc);
                        return 2.0f * a.grad_scale * d;
                    };
                    auto cterm = [&](float x, float c) {   // COT: adds x * c, returns the scaled cotangent entry
                        loss_acc = fmaf(x, c, loss_acc);
                        return a.grad_scale * c;
                    };
                    Row<CE> g = zero_row<CE>();
                    if (a.dim == 2) {
                        // 2-D meshes: float2 rows, no per-channel tests; the channels beyond dim have d = 0, whose
                        // loss term (+0) and cotangent (0) the general form below would add
                        if (a.x_phys) *reinterpret_cast<float2*>(a.x_phys + gi * 2) = make_float2(xn.v[0], xn.v[1]);
                        const float2 tg = stage ? *reinterpret_cast<const float2*>(DL + (size_t)i * 8)
                                                : *reinterpret_cast<const float2*>(a.target + gi * 2);
                        if constexpr (COT) {
                            g.v[0] = cterm(xn.v[0], tg.x);
                            g.v[1] = cterm(xn.v[1], tg.y);
                        } else {
                            g.v[0] = term(xn.v[0] - tg.x);
                            g.v[1] = term(xn.v[1] - tg.y);
                        }
                    } else {
                        if (a.x_phys) store_dims<CE>(a.x_phys, gi, a.dim, xn);
                        const Row<CE> tg = stage ? load_dims<CE>(reinterpret_cast<const float*>(TG + i * tg_rb), 0, a.dim)
                                                 : load_dims<CE>(a.target, gi, a.dim);
                        if constexpr (COT) {
#pragma unroll
                            for (int c = 0; c < CE; ++c) g.v[c] = cterm(xn.v[c], tg.v[c]);   // load_dims: 0 beyond dim
                        } else {
#pragma unroll
                            for (int c = 0; c < CE; ++c) g.v[c] = term((c < a.dim) ? xn.v[c] - tg.v[c] : 0.f);
                        }
                    }
                    return g;
                };
                const Row<CE> p = project<CE>(Mu, y);
                if (src) sts_row<CE>(P, i * RB, p);
                Row<CE> gp, t, o;
                float D, lse;
                ell_feval_bwd_dst<CE, W>(Xc, e, y, p, h, cot, gp, D, lse, t, o);
                // the rest of tile_backward's phase A at xi = y, b = h
                if (need_gtau) {
#pragma unroll
                    for (int c = 0; c < CE; ++c) gtau = fmaf(gp.v[c], o.v[c] - y.v[c], gtau);
                }
#pragma unroll
                for (int aa = 0; aa < CE; ++aa)
#pragma unroll
                    for (int bb = 0; bb < CE; ++bb) acc[aa * CE + bb] = fmaf(y.v[aa], t.v[bb], acc[aa * CE + bb]);
#pragma unroll
                for (int bb = 0; bb < CE; ++bb) acc[CE * CE + bb] += t.v[bb];
                if (src) {
                    const Row<CE> Mt = apply_M<CE>(Mu, t);
                    Row<CE> go, gs;
#pragma unroll
                    for (int c = 0; c < CE; ++c) {
                        go.v[c] = h * gp.v[c];
                        gs.v[c] = fmaf(1.0f - h, gp.v[c], Mt.v[c]);   // Euler: a = 1
                    }
                    // at dim 2 the DL row of node i held node i's staged target, read above by this thread only
                    *reinterpret_cast<float2*>(DL + (size_t)i * 8) = make_float2(D, lse);
                    sts_row<CE>(Xn, i * RB, go);
                    sts_row<CE>(GS, i * RB, gs);
                }
            }
            // the tile's loss: warp sums before the barrier that ends the layer, the cross-warp sum after it
            float one[1] = {loss_acc};
            block_reduce_warps<1>(one, red);
            __syncthreads();
            tr.mark();   // 2+L: last forward layer + phase A of its backward
            block_reduce_finish<1>(red, a.loss_partials + tile);
            if (!src) __syncthreads();   // the block reduction that follows at once reuses `red`
            tr.mark();   // loss reduced
            tile_backward<CE, W, ELLS, true>(a, tile, n0, NT, Xc, Xn, P, DL, GS, Ein, Eout, Mu, red, acc, gtau);
            tr.mark();   // backward + block reduction done
        }
        } else {
        // ---- forward (RK4 steps), loss and cotangent fused into stage 4 of the last step ----------
        unsigned char* XB = P;    // base state of the step
        unsigned char* AC = GS;   // k-accumulator
        unsigned char* G = smem + lay.g;
        float loss_acc = 0.f;
        for (int l = 0; l < a.L; ++l) {
            if (a.Lw > 1 && l > 0) {
                for (int t = tid; t < MUSZ; t += nthr) Mu[t] = a.Mu[(size_t)l * MUSZ + t];
                __syncthreads();
            }
            const float h = __ldcg(a.tau + l);
            const bool last = (l == a.L - 1);
            float* st_out = last ? nullptr : a.states + (size_t)(l + 1) * state_stride;
            const float cin[4] = {0.5f * h, 0.5f * h, h, 0.f};
            const float wacc[4] = {1.f, 2.f, 2.f, 1.f};
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                for (int i = tid; i < NT; i += nthr) {
                    const uint4 e = Ein.get(i);
                    const Row<CE> y = lds_row<CE>(Xc, i * RB);
                    if (l == 0 && s == 0) store_row<CE>(a.states, (int64_t)n0 + i, y);
                    const Row<CE> k = ell_feval<CE, W>(Xc, e, y, Mu);
                    Row<CE> base, acc, out;
                    if (s == 0) {
                        base = y;
                        acc = k;
                        sts_row<CE>(XB, i * RB, y);
                    } else {
                        base = lds_row<CE>(XB, i * RB);
                        acc = lds_row<CE>(AC, i * RB);
#pragma unroll
                        for (int c = 0; c < CE; ++c) acc.v[c] = fmaf(wacc[s], k.v[c], acc.v[c]);
                    }
                    if (s < 3) {
                        sts_row<CE>(AC, i * RB, acc);
#pragma unroll
                        for (int c = 0; c < CE; ++c) out.v[c] = fmaf(cin[s], k.v[c], base.v[c]);
                        sts_row<CE>(Xn, i * RB, out);
                    } else {
#pragma unroll
                        for (int c = 0; c < CE; ++c) out.v[c] = fmaf(h * (1.0f / 6.0f), acc.v[c], base.v[c]);
                        if (!last) {
                            sts_row<CE>(Xn, i * RB, out);
                            store_row<CE>(st_out, (int64_t)n0 + i, out);
                        } else {
                            const int64_t gi = (int64_t)n0 + i;
                            if (a.x_phys) store_dims<CE>(a.x_phys, gi, a.dim, out);
                            const Row<CE> tg = stage ? load_dims<CE>(reinterpret_cast<const float*>(DL), i, a.dim)
                                                     : load_dims<CE>(a.target, gi, a.dim);
                            Row<CE> g;
#pragma unroll
                            for (int c = 0; c < CE; ++c) {
                                if constexpr (COT) {
                                    const float cc = (c < a.dim) ? tg.v[c] : 0.f;
                                    loss_acc = fmaf(out.v[c], cc, loss_acc);
                                    g.v[c] = a.grad_scale * cc;
                                } else {
                                    const float d = (c < a.dim) ? out.v[c] - tg.v[c] : 0.f;
                                    if (a.loss_kind == 0) {
                                        loss_acc += fabsf(d);
                                        g.v[c] = (d > 0.f) ? a.grad_scale : ((d < 0.f) ? -a.grad_scale : 0.f);   // torch sign()
                                    } else {
                                        loss_acc = fmaf(d, d, loss_acc);
                                        g.v[c] = 2.0f * a.grad_scale * d;
                                    }
                                }
                            }
                            sts_row<CE>(G, i * RB, g);
                        }
                    }
                }
                __syncthreads();
                unsigned char* t = Xc;
                Xc = Xn;
                Xn = t;
            }
            tr.mark();   // 3 .. 2+L: forward steps
        }
        {
            float one[1] = {loss_acc};
            block_reduce<1>(one, red, a.loss_partials + tile);
        }
        tr.mark();   // loss reduced
        tile_backward_rk4<CE, W, ELLS>(a, tile, n0, NT, smem, lay, Ein, Eout, Mu, red);
        tr.mark();   // backward + block reduction done
        }
    }

    // ---- tail: the last CTA to finish reduces the partials (fixed order -> deterministic), applies
    // the chain rule to the Linear parameters and, single-GPU, takes the Adam step and refolds the
    // weights for the next launch: the whole training step is this one kernel.
    if (a.tail == 0) return;
    if (!reducer) {
        // every global value the tail reads (partials, loss / step-size partials) was written by warp 0
        // (block_reduce): release them with one fence, then count this CTA in
        if (tid < 32) {
            __threadfence();
            __syncwarp();
            if (tid == 0) {
                const unsigned int prev = atomicAdd(a.counter, 1u);
                s_last = (prev == gridDim.x - 1) ? 1 : 0;
            }
        }
        if (a.tail_cta) return;
        __syncthreads();
        if (!s_last) return;
        tr.mark();   // elected
    }
    TailCtx cx;
    if (reducer) pdl_wait();   // previous step complete: its step counter, moments and weights are final
    tail_prepare<CE>(a, smem, lay.bar, cx);
    if (reducer) {
        tr.mark();   // prepared
        if (a.tail >= 2 && tid == nthr - 1) {
            s_step = __ldcg(a.step) + 1;
            s_coef = tail::adam_coef(a.lr, a.beta1, a.beta2, a.eps, a.weight_decay, a.adam_grad_scale, s_step);
        }
        if (tid == 0) {
            unsigned int seen;
            do {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.counter) : "memory");
            } while (seen < (unsigned)tile_ctas);
        }
        __syncthreads();
        tr.mark();   // every tile CTA has checked in
    }
    __threadfence();
    tail_finish<CE>(a, smem, cx, s_coef, s_step, tr);
    if (tid == 0) *a.counter = 0u;
    tr.mark();   // tail done
}

// ============================================================================================
// host-side launchers (instantiated per (CE, W) translation unit by GAD_ELL_INSTANTIATE)
// ============================================================================================
template <typename K>
int prepare_launch(K kernel, int threads, size_t smem_bytes, int T, int* grid) {
    GAD_CHECK_ARG((int)smem_bytes <= smem_optin_bytes(), "ELL kernel: tile needs %zu B of shared memory (> %d)",
                  smem_bytes, smem_optin_bytes());
    GAD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    GAD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    int occ = 0;
    GAD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem_bytes));
    GAD_CHECK_ARG(occ >= 1, "ELL kernel: launch of %d threads with %zu B of shared memory does not fit an SM", threads,
                  smem_bytes);
    const long long cap = (long long)occ * sm_count();
    *grid = (int)((long long)T < cap ? T : cap);
    return GAD_OK;
}

template <int CE, int W, bool ELLS>
int launch_fwd_t(const Args& a, int method, int threads, cudaStream_t st) {
    int grid = 0, rc;
    if (method == GAD_METHOD_EULER) {
        const size_t bytes = make_layout(CE, KIND_FWD, a.cap_nodes, ELLS, (threads + 31) / 32).total;
        if ((rc = prepare_launch(k_ell_fwd<CE, W, ELLS, GAD_METHOD_EULER>, threads, bytes, a.T, &grid))) return rc;
        k_ell_fwd<CE, W, ELLS, GAD_METHOD_EULER><<<grid, threads, bytes, st>>>(a);
    } else {
        const size_t bytes = make_layout(CE, KIND_FWD_RK4, a.cap_nodes, ELLS, (threads + 31) / 32).total;
        if ((rc = prepare_launch(k_ell_fwd<CE, W, ELLS, GAD_METHOD_RK4>, threads, bytes, a.T, &grid))) return rc;
        k_ell_fwd<CE, W, ELLS, GAD_METHOD_RK4><<<grid, threads, bytes, st>>>(a);
    }
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

template <int CE, int W, bool ELLS>
int launch_bwd_t(const Args& a, int threads, cudaStream_t st) {
    int grid = 0, rc;
    const size_t bytes = make_layout(CE, KIND_BWD, a.cap_nodes, ELLS, (threads + 31) / 32).total;
    if ((rc = prepare_launch(k_ell_bwd<CE, W, ELLS>, threads, bytes, a.T, &grid))) return rc;
    k_ell_bwd<CE, W, ELLS><<<grid, threads, bytes, st>>>(a);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

template <int CE, int W, bool ELLS>
int launch_bwd_rk4_t(const Args& a, int threads, cudaStream_t st) {
    int grid = 0, rc;
    const size_t bytes = make_layout(CE, KIND_BWD_RK4, a.cap_nodes, ELLS, (threads + 31) / 32).total;
    if ((rc = prepare_launch(k_ell_bwd_rk4<CE, W, ELLS>, threads, bytes, a.T, &grid))) return rc;
    k_ell_bwd_rk4<CE, W, ELLS><<<grid, threads, bytes, st>>>(a);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

template <int CE, int W, bool ELLS, int METHOD, bool COT>
int launch_train_m(const Args& a_in, int threads, cudaStream_t st) {
    int grid = 0, rc;
    const int kind = METHOD == GAD_METHOD_RK4 ? KIND_TRAIN_RK4 : KIND_BWD;
    const size_t bytes = make_layout(CE, kind, a_in.cap_nodes, ELLS, (threads + 31) / 32).total;
    if ((rc = prepare_launch(k_ell_train<CE, W, ELLS, METHOD, COT>, threads, bytes, a_in.T + 1, &grid))) return rc;
    Args a = a_in;
    // grid == T + 1: every tile has its own CTA and one more fits -> that one is the reducer
    static const bool allow_reducer = !(getenv("GAD_TAIL_CTA") && atoi(getenv("GAD_TAIL_CTA")) == 0);
    a.tail_cta = (allow_reducer && a.tail != 0 && grid == a.T + 1) ? 1 : 0;
    if (!a.tail_cta && grid > a.T) grid = a.T;
    if (a.pdl) {
        // programmatic dependent launch: this kernel may start while its predecessor in the stream is
        // still running (it synchronises itself with griddepcontrol.wait)
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3((unsigned)threads);
        cfg.dynamicSmemBytes = bytes;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        GAD_CUDA(cudaLaunchKernelEx(&cfg, k_ell_train<CE, W, ELLS, METHOD, COT>, a));
        count_launch(1);
        return GAD_OK;
    }
    k_ell_train<CE, W, ELLS, METHOD, COT><<<grid, threads, bytes, st>>>(a);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

template <int CE, int W, bool ELLS>
int launch_train_t(const Args& a, int method, int threads, cudaStream_t st) {
    if (a.loss_kind == 2) {
        if (method == GAD_METHOD_RK4) return launch_train_m<CE, W, ELLS, GAD_METHOD_RK4, true>(a, threads, st);
        return launch_train_m<CE, W, ELLS, GAD_METHOD_EULER, true>(a, threads, st);
    }
    if (method == GAD_METHOD_RK4) return launch_train_m<CE, W, ELLS, GAD_METHOD_RK4, false>(a, threads, st);
    return launch_train_m<CE, W, ELLS, GAD_METHOD_EULER, false>(a, threads, st);
}

// which: 0 forward, 1 backward, 2 train (Euler or RK4 by `method`), 3 backward through RK4 steps
#define GAD_ELL_INSTANTIATE(CE_, W_)                                                                         \
    int ell_launch_c##CE_##w##W_(int which, const Args& a, int method, int ells, int threads, cudaStream_t st) { \
        if (which == 3)                                                                                      \
            return ells ? launch_bwd_rk4_t<CE_, W_, true>(a, threads, st) : launch_bwd_rk4_t<CE_, W_, false>(a, threads, st); \
        if (which == 0)                                                                                      \
            return ells ? launch_fwd_t<CE_, W_, true>(a, method, threads, st)                                \
                        : launch_fwd_t<CE_, W_, false>(a, method, threads, st);                              \
        if (which == 1)                                                                                      \
            return ells ? launch_bwd_t<CE_, W_, true>(a, threads, st) : launch_bwd_t<CE_, W_, false>(a, threads, st); \
        return ells ? launch_train_t<CE_, W_, true>(a, method, threads, st)                                 \
                    : launch_train_t<CE_, W_, false>(a, method, threads, st);                               \
    }

#define GAD_ELL_DECLARE(CE_, W_) \
    int ell_launch_c##CE_##w##W_(int which, const Args& a, int method, int ells, int threads, cudaStream_t st);

}  // namespace ell
}  // namespace gad
