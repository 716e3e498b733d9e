// Per-node arithmetic of one attention-diffusion F-evaluation and of its backward, shared by the
// streaming kernels (state in global memory / L2) and the mesh-resident kernels (state in shared
// memory).  Everything is templated on CE, the number of live channels (2, 4, 8), so a node row is
// one or two 128-bit (or one 64-bit) accesses.
//
// Forward, per destination node i (src/GRAND_plus.py:225-343 with value = identity):
//     p_i   = M^T x_i + u                          (folded q/k projection, see weights.cu)
//     s_e   = <p_i, x_j>                           for every in-edge e = (j -> i), CSR row order
//     m_i   = max_e s_e,  w_e = exp(s_e - m_i),  Z_i = sum_e w_e
//     o_i   = (sum_e w_e x_j) / Z_i                (= sum_e alpha_e x_j, alpha row-stochastic)
//     k_i   = o_i - x_i                            (GRAND_plus.py:267)
// Z_i >= 1 in fp32, so the reference's "+1e-16" (PyG softmax) is a no-op and is dropped.
// A node without in-edges gets o_i = 0 (empty scatter row), exactly like the reference.
//
// Backward (SURVEY A.2, re-derived for the folded form), with g_o = b * g_plus:
//     D_i = <g_o, o_i>;  da_e = <g_o, x_j>;  ds_e = alpha_e (da_e - D_i);  t_i = sum_e ds_e x_j
//     G_M += x_i (x) t_i;  G_u += t_i;  g_x[i] += M t_i                      (destination pass)
//     g_x[j] += alpha_e g_o[i] + ds_e p_i                                    (source pass)
//
// Row caching.  Mesh rows are short (in-degree <= 7), so a row of up to GAD_ROW_W neighbours is
// gathered ONCE into registers (all gathers issued back to back -> memory-level parallelism) and
// max / exp / aggregate / backward terms are computed from registers; longer rows fall back to
// multi-pass loops over the row.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

// ---- build-time variant switches (defaults = shipped configuration) -------------------------
#ifndef GAD_FAST_EXP
#define GAD_FAST_EXP 0      // 1: ex2.approx-based __expf instead of expf
#endif
#ifndef GAD_ROW_W
#define GAD_ROW_W 0         // register-cached row width; 0 disables row caching (measured: slower at 127 regs)
#endif
#ifndef GAD_BWD_ROWCACHE
#define GAD_BWD_ROWCACHE 1  // destination pass of the backward also row-cached
#endif

namespace gad {

// All logits are in the log2 domain: gad_prepare_weights folds log2(e) into (M, u), so
// alpha_e = 2^(s_e - m) / Z and the backward carries ds' = ln2 * alpha (da - D); gad_weight_grads
// undoes the fold.  ex2.approx / lg2.approx are single MUFU ops with 2^-22 relative error.
constexpr float LN2_F = 0.69314718055994530942f;

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// rcp.approx + one Newton step.  The raw MUFU result is off by up to 2^-22 with a SYSTEMATIC sign, so
// the attention weights of a row would sum to 1 + eps with the same eps at every node; in the
// backward that leaves sum_e ds_e = -ln2 eps D_i instead of 0, a bias that does not average out in
// G_u = sum_i t_i (the gradient of lin_query.bias), whose true value is a heavily cancelling sum.
// Two FMAs bring the weights' sum to 1 within rounding (random sign).
__device__ __forceinline__ float rcp_refined(float x) {
    const float r = rcp_approx(x);
    return fmaf(r, fmaf(-x, r, 1.0f), r);
}
__device__ __forceinline__ float gexp(float x) { return ex2_approx(x); }

template <int CE>
struct Row {
    float v[CE];
};

template <int CE>
__device__ __forceinline__ Row<CE> zero_row() {
    Row<CE> r;
#pragma unroll
    for (int c = 0; c < CE; ++c) r.v[c] = 0.f;
    return r;
}

template <int CE>
__device__ __forceinline__ Row<CE> load_row(const float* __restrict__ base, int64_t i) {
    Row<CE> r;
    if constexpr (CE == 2) {
        const float2 t = *reinterpret_cast<const float2*>(base + i * 2);
        r.v[0] = t.x;
        r.v[1] = t.y;
    } else {
#pragma unroll
        for (int q = 0; q < CE / 4; ++q) {
            const float4 t = *reinterpret_cast<const float4*>(base + i * CE + 4 * q);
            r.v[4 * q + 0] = t.x;
            r.v[4 * q + 1] = t.y;
            r.v[4 * q + 2] = t.z;
            r.v[4 * q + 3] = t.w;
        }
    }
    return r;
}

template <int CE>
__device__ __forceinline__ void store_row(float* __restrict__ base, int64_t i, const Row<CE>& r) {
    if constexpr (CE == 2) {
        *reinterpret_cast<float2*>(base + i * 2) = make_float2(r.v[0], r.v[1]);
    } else {
#pragma unroll
        for (int q = 0; q < CE / 4; ++q)
            *reinterpret_cast<float4*>(base + i * CE + 4 * q) =
                make_float4(r.v[4 * q], r.v[4 * q + 1], r.v[4 * q + 2], r.v[4 * q + 3]);
    }
}

template <int CE>
__device__ __forceinline__ float dot(const Row<CE>& a, const Row<CE>& b) {
    float s = a.v[0] * b.v[0];
#pragma unroll
    for (int c = 1; c < CE; ++c) s = fmaf(a.v[c], b.v[c], s);
    return s;
}

// p = M^T x + u   (M row-major [a][b], Mu = {M, u})
template <int CE>
__device__ __forceinline__ Row<CE> project(const float* __restrict__ Mu, const Row<CE>& x) {
    Row<CE> p;
#pragma unroll
    for (int b = 0; b < CE; ++b) p.v[b] = Mu[CE * CE + b];
#pragma unroll
    for (int a = 0; a < CE; ++a)
#pragma unroll
        for (int b = 0; b < CE; ++b) p.v[b] = fmaf(x.v[a], Mu[a * CE + b], p.v[b]);
    return p;
}

// p = M^T y + u with the per-mesh offset of the folded bias (global CNN features, include/gadapt.h): `dui` = the CE
// floats du[mesh, lw] of the node's mesh, or null.  u + du is rounded before the products are added, as the mesh-resident
// kernels do when they fold du into their shared copy of u (ell_kernels.cuh: load_mu), so every route rounds alike.
template <int CE>
__device__ __forceinline__ Row<CE> project_du(const float* __restrict__ Mu, const float* __restrict__ dui, const Row<CE>& x) {
    if (!dui) return project<CE>(Mu, x);
    Row<CE> p;
#pragma unroll
    for (int b = 0; b < CE; ++b) p.v[b] = Mu[CE * CE + b] + __ldg(dui + b);
#pragma unroll
    for (int a = 0; a < CE; ++a)
#pragma unroll
        for (int b = 0; b < CE; ++b) p.v[b] = fmaf(x.v[a], Mu[a * CE + b], p.v[b]);
    return p;
}

// y = M t
template <int CE>
__device__ __forceinline__ Row<CE> apply_M(const float* __restrict__ Mu, const Row<CE>& t) {
    Row<CE> y;
#pragma unroll
    for (int a = 0; a < CE; ++a) {
        float s = 0.f;
#pragma unroll
        for (int b = 0; b < CE; ++b) s = fmaf(Mu[a * CE + b], t.v[b], s);
        y.v[a] = s;
    }
    return y;
}

struct SoftmaxStats {
    float m;    // row max of the logits (0 for an empty row)
    float rZ;   // 1 / sum exp(s - m)    (0 for an empty row)
};

// Rows longer than the register cache (and builds with GAD_ROW_W == 0) use the row-cached code
// only when CE * GAD_ROW_W registers are affordable: CE = 8 keeps the multi-pass loops.
template <int CE>
struct RowCache {
    static constexpr int W = (CE <= 4) ? GAD_ROW_W : 0;
};

// One F-evaluation at node i.  X: state rows (global or shared), indexed by the entries of `col`
// (already relative to X).  Returns k_i = o_i - x_i; o_i, the softmax stats and p_i on request.
// dui: the bias offset of node i's mesh (project_du), or null.
template <int CE, typename ColT>
__device__ __forceinline__ Row<CE> node_feval(const float* __restrict__ X, const ColT* __restrict__ col,
                                              int e_begin, int e_end, const Row<CE>& xi,
                                              const float* __restrict__ Mu, Row<CE>* o_out = nullptr,
                                              SoftmaxStats* st_out = nullptr, Row<CE>* p_out = nullptr,
                                              const float* __restrict__ dui = nullptr) {
    const Row<CE> p = project_du<CE>(Mu, dui, xi);
    const int deg = e_end - e_begin;
    float m = -CUDART_INF_F, Z = 0.f;
    Row<CE> o = zero_row<CE>();
    constexpr int W = RowCache<CE>::W;
    if (W > 0 && deg <= W) {
        Row<CE> xj[W > 0 ? W : 1];
        float s[W > 0 ? W : 1];
#pragma unroll
        for (int q = 0; q < W; ++q) {
            if (q < deg) {
                xj[q] = load_row<CE>(X, (int64_t)col[e_begin + q]);
                s[q] = dot<CE>(p, xj[q]);
                m = fmaxf(m, s[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < W; ++q) {
            if (q < deg) {
                const float w = gexp(s[q] - m);
                Z += w;
#pragma unroll
                for (int c = 0; c < CE; ++c) o.v[c] = fmaf(w, xj[q].v[c], o.v[c]);
            }
        }
    } else {
        for (int e = e_begin; e < e_end; ++e) {
            const Row<CE> xj = load_row<CE>(X, (int64_t)col[e]);
            m = fmaxf(m, dot<CE>(p, xj));
        }
        for (int e = e_begin; e < e_end; ++e) {
            const Row<CE> xj = load_row<CE>(X, (int64_t)col[e]);
            const float w = gexp(dot<CE>(p, xj) - m);
            Z += w;
#pragma unroll
            for (int c = 0; c < CE; ++c) o.v[c] = fmaf(w, xj.v[c], o.v[c]);
        }
    }
    const float rZ = (deg > 0) ? 1.0f / Z : 0.f;
    Row<CE> k;
#pragma unroll
    for (int c = 0; c < CE; ++c) {
        o.v[c] *= rZ;
        k.v[c] = o.v[c] - xi.v[c];
    }
    if (o_out) *o_out = o;
    if (st_out) {
        st_out->m = (deg > 0) ? m : 0.f;
        st_out->rZ = rZ;
    }
    if (p_out) *p_out = p;
    return k;
}

// Per-destination record the source pass needs: p_i, D_i and the log-sum-exp of row i.
template <int CE>
struct DstRec {
    Row<CE> p;
    float D;
    float lse;
};

// Destination pass of the backward at node i.
//   gplus = dL/dx^{l+1}_i,  a, b: x^{l+1} = a x + b (o - x)  (Euler: a = 1, b = tau)
// Returns the part of dL/dx^l_i that is local to row i:  (a - b) gplus + M t_i.
// Accumulates G_M (x) / G_u into acc[CE*CE + CE] and  <gplus, o - x>  into *gb_acc.
template <int CE, typename ColT>
__device__ __forceinline__ Row<CE> node_bwd_dst(const float* __restrict__ X, const ColT* __restrict__ col,
                                                int e_begin, int e_end, const Row<CE>& xi,
                                                const Row<CE>& gplus, float a, float b,
                                                const float* __restrict__ Mu, DstRec<CE>* rec,
                                                float* __restrict__ acc, float* gb_acc) {
    const int deg = e_end - e_begin;
    Row<CE> go;
#pragma unroll
    for (int c = 0; c < CE; ++c) go.v[c] = b * gplus.v[c];
    Row<CE> t = zero_row<CE>();
    Row<CE> p, o;
    float D, m, rZ;
    constexpr int W = GAD_BWD_ROWCACHE ? RowCache<CE>::W : 0;
    if (W > 0 && deg <= W) {
        p = project<CE>(Mu, xi);
        Row<CE> xj[W > 0 ? W : 1];
        float s[W > 0 ? W : 1], da[W > 0 ? W : 1];
        m = -CUDART_INF_F;
#pragma unroll
        for (int q = 0; q < W; ++q) {
            if (q < deg) {
                xj[q] = load_row<CE>(X, (int64_t)col[e_begin + q]);
                s[q] = dot<CE>(p, xj[q]);
                da[q] = dot<CE>(go, xj[q]);
                m = fmaxf(m, s[q]);
            }
        }
        float Z = 0.f;
        o = zero_row<CE>();
#pragma unroll
        for (int q = 0; q < W; ++q) {
            if (q < deg) {
                s[q] = gexp(s[q] - m);          // s[q] now holds w_q
                Z += s[q];
#pragma unroll
                for (int c = 0; c < CE; ++c) o.v[c] = fmaf(s[q], xj[q].v[c], o.v[c]);
            }
        }
        rZ = (deg > 0) ? 1.0f / Z : 0.f;
#pragma unroll
        for (int c = 0; c < CE; ++c) o.v[c] *= rZ;
        D = dot<CE>(go, o);
#pragma unroll
        for (int q = 0; q < W; ++q) {
            if (q < deg) {
                const float ds = (s[q] * rZ * LN2_F) * (da[q] - D);
#pragma unroll
                for (int c = 0; c < CE; ++c) t.v[c] = fmaf(ds, xj[q].v[c], t.v[c]);
            }
        }
        if (deg == 0) m = 0.f;
    } else {
        SoftmaxStats st;
        node_feval<CE, ColT>(X, col, e_begin, e_end, xi, Mu, &o, &st, &p);
        m = st.m;
        rZ = st.rZ;
        D = dot<CE>(go, o);
        for (int e = e_begin; e < e_end; ++e) {
            const Row<CE> xj = load_row<CE>(X, (int64_t)col[e]);
            const float alpha = gexp(dot<CE>(p, xj) - m) * rZ;
            const float ds = (alpha * LN2_F) * (dot<CE>(go, xj) - D);
#pragma unroll
            for (int c = 0; c < CE; ++c) t.v[c] = fmaf(ds, xj.v[c], t.v[c]);
        }
    }
    float gb = 0.f;
#pragma unroll
    for (int c = 0; c < CE; ++c) gb = fmaf(gplus.v[c], o.v[c] - xi.v[c], gb);
    *gb_acc += gb;
#pragma unroll
    for (int aa = 0; aa < CE; ++aa)
#pragma unroll
        for (int bb = 0; bb < CE; ++bb) acc[aa * CE + bb] = fmaf(xi.v[aa], t.v[bb], acc[aa * CE + bb]);
#pragma unroll
    for (int bb = 0; bb < CE; ++bb) acc[CE * CE + bb] += t.v[bb];
    rec->p = p;
    rec->D = D;
    // alpha_e = 2^(s_e - lse);  lse = m + log2 Z.  Empty row: never read by a source pass.
    rec->lse = (deg > 0) ? m - log2f(rZ) : 0.f;
    const Row<CE> Mt = apply_M<CE>(Mu, t);
    Row<CE> gs;
#pragma unroll
    for (int c = 0; c < CE; ++c) gs.v[c] = fmaf(a - b, gplus.v[c], Mt.v[c]);
    return gs;
}

// Source pass of the backward at node j: contributions of all out-edges (j -> i).
//   P: rows p_i;  DL: float2 rows (D_i, lse_i);  G: rows gplus_i;  tdst: destinations, CSC order.
template <int CE, typename ColT>
__device__ __forceinline__ Row<CE> node_bwd_src(const float* __restrict__ P, const float2* __restrict__ DL,
                                                const float* __restrict__ G, const ColT* __restrict__ tdst,
                                                int e_begin, int e_end, const Row<CE>& xj, float b) {
    Row<CE> accv = zero_row<CE>();
#pragma unroll 2
    for (int e = e_begin; e < e_end; ++e) {
        const int64_t i = (int64_t)tdst[e];
        const Row<CE> p = load_row<CE>(P, i);
        const Row<CE> gp = load_row<CE>(G, i);
        const float2 dl = DL[i];
        const float alpha = gexp(dot<CE>(p, xj) - dl.y);
        const float da = b * dot<CE>(gp, xj);
        const float ds = (alpha * LN2_F) * (da - dl.x);
        const float ab = alpha * b;
#pragma unroll
        for (int c = 0; c < CE; ++c) accv.v[c] = fmaf(ab, gp.v[c], fmaf(ds, p.v[c], accv.v[c]));
    }
    return accv;
}

// Deterministic block-wide sum of NACC per-thread accumulators into out[0..NACC).
// red must hold NACC * (blockDim/32) floats.  The two halves are also called on their own by a
// caller that already has a barrier between them (and keeps `red` untouched until the second is done).
template <int NACC>
__device__ __forceinline__ void block_reduce_warps(const float (&acc)[NACC], float* __restrict__ red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
        float v = acc[k];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        if (lane == 0) red[k * nwarp + warp] = v;
    }
}

template <int NACC>
__device__ __forceinline__ void block_reduce_finish(const float* __restrict__ red, float* __restrict__ out) {
    const int nwarp = (blockDim.x + 31) >> 5;
    for (int k = threadIdx.x; k < NACC; k += blockDim.x) {
        double s = 0.0;   // the sums cancel heavily (signed gradient terms): keep the cross-warp step exact
        for (int w = 0; w < nwarp; ++w) s += (double)red[k * nwarp + w];
        out[k] = (float)s;
    }
}

template <int NACC>
__device__ __forceinline__ void block_reduce(float (&acc)[NACC], float* __restrict__ red,
                                             float* __restrict__ out) {
    block_reduce_warps<NACC>(acc, red);
    __syncthreads();
    block_reduce_finish<NACC>(red, out);
    __syncthreads();
}

}  // namespace gad
