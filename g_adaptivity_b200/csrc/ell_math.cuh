// ELL-row node arithmetic for the mesh-resident kernels (ell_kernels.cuh).
//
// Mesh graphs have tiny, bounded degree (<= 7 incoming / outgoing edges per node, self-loops
// included), so a tile's topology is stored as fixed-width rows of eight uint16:
//     ell[i] = { off_0 .. off_6, valid }    off_q = (tile-local index of the row in slot q) * ROWBYTES
// One 128-bit load fetches a node's whole adjacency; the offsets are pre-multiplied byte offsets
// into the shared-memory state buffer, so a neighbour gather is `LDS.128 [off + base]` with no
// address arithmetic.  Bit q of `valid` says slot q holds a neighbour; the other slots point at a
// valid row too and are masked out of the softmax by setting their logit to -inf, which makes
// every per-slot code path branch-free: all W gathers of a row are issued back to back
// (memory-level parallelism), then max / ex2 / aggregate run from registers.  The builder
// (ell_api.cu: k_build_ell) gives every neighbour offset its own slot, so the q-th gather of
// consecutive lanes reads consecutive rows on structured meshes.
//
// All logits are in the log2 domain: gad_prepare_weights folds log2(e) into (M, u), the kernels
// use ex2.approx / lg2.approx / rcp.approx (one MUFU each, relative error 2^-22), and the backward
// carries the matching ln 2 factor (ds' = ln2 * alpha * (da - D) = dL/ds'); gad_weight_grads
// differentiates through the fold.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "node_math.cuh"

namespace gad {

constexpr int ELL_SLOTS = 7;      // neighbour slots per row; the 8th uint16 is the validity mask

template <int CE>
struct EllRow {
    static constexpr uint32_t BYTES = CE * sizeof(float);   // ROWBYTES: 8 (CE = 2) or 16 (CE = 4)
};

__device__ __forceinline__ uint32_t ell_off(const uint4& e, int q) {
    const uint32_t w = (q >> 1) == 0 ? e.x : ((q >> 1) == 1 ? e.y : ((q >> 1) == 2 ? e.z : e.w));
    return (q & 1) ? (w >> 16) : (w & 0xffffu);
}
__device__ __forceinline__ uint32_t ell_valid(const uint4& e) { return e.w >> 16; }
__device__ __forceinline__ bool ell_has(const uint4& e, int q) { return (e.w >> (16 + q)) & 1u; }

template <int CE>
__device__ __forceinline__ Row<CE> lds_row(const unsigned char* __restrict__ base, uint32_t byte_off) {
    Row<CE> r;
    if constexpr (CE == 2) {
        const float2 t = *reinterpret_cast<const float2*>(base + byte_off);
        r.v[0] = t.x;
        r.v[1] = t.y;
    } else {
        const float4 t = *reinterpret_cast<const float4*>(base + byte_off);
        r.v[0] = t.x;
        r.v[1] = t.y;
        r.v[2] = t.z;
        r.v[3] = t.w;
    }
    return r;
}

template <int CE>
__device__ __forceinline__ void sts_row(unsigned char* __restrict__ base, uint32_t byte_off, const Row<CE>& r) {
    if constexpr (CE == 2) {
        *reinterpret_cast<float2*>(base + byte_off) = make_float2(r.v[0], r.v[1]);
    } else {
        *reinterpret_cast<float4*>(base + byte_off) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
    }
}

// ---- forward: k = F(y) = A(y) y - y at one node ------------------------------------------------
// Xb: state buffer (bytes), ell: the node's in-adjacency row, y: the node's own state.
template <int CE, int W>
__device__ __forceinline__ Row<CE> ell_feval(const unsigned char* __restrict__ Xb, const uint4& ell,
                                             const Row<CE>& y, const float* __restrict__ Mu) {
    const bool any = ell_valid(ell) != 0;
    const Row<CE> p = project<CE>(Mu, y);
    Row<CE> xj[W];
    float s[W];
    float m = -3.0e38f;   // finite floor: an empty row gives w = 2^(-inf) = 0 instead of NaN
#pragma unroll
    for (int q = 0; q < W; ++q) {
        xj[q] = lds_row<CE>(Xb, ell_off(ell, q));
        const float d = dot<CE>(p, xj[q]);
        s[q] = ell_has(ell, q) ? d : -CUDART_INF_F;
        m = fmaxf(m, s[q]);
    }
    float Z = 0.f;
    Row<CE> o = zero_row<CE>();
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const float w = ex2_approx(s[q] - m);
        Z += w;
#pragma unroll
        for (int c = 0; c < CE; ++c) o.v[c] = fmaf(w, xj[q].v[c], o.v[c]);
    }
    const float rZ = any ? rcp_refined(Z) : 0.f;   // no in-edge: o = 0 (empty scatter row)
    Row<CE> k;
#pragma unroll
    for (int c = 0; c < CE; ++c) k.v[c] = fmaf(o.v[c], rZ, -y.v[c]);
    return k;
}

// ---- backward, destination pass -------------------------------------------------------------
// Inputs: own state x_i, go = b * gplus_i.  Outputs: p_i (log2 domain), D_i = <go, o_i>,
// lse_i (log2), t_i = sum_e ds'_e x_j with ds'_e = ln2 alpha_e (<go, x_j> - D_i), and o_i.
template <int CE, int W>
__device__ __forceinline__ void ell_bwd_dst(const unsigned char* __restrict__ Xb, const uint4& ell,
                                            const Row<CE>& xi, const Row<CE>& go, const float* __restrict__ Mu,
                                            Row<CE>& p, float& D, float& lse, Row<CE>& t, Row<CE>& o) {
    const bool any = ell_valid(ell) != 0;
    p = project<CE>(Mu, xi);
    Row<CE> xj[W];
    float s[W];
    float m = -3.0e38f;
#pragma unroll
    for (int q = 0; q < W; ++q) {
        xj[q] = lds_row<CE>(Xb, ell_off(ell, q));
        const float d = dot<CE>(p, xj[q]);
        s[q] = ell_has(ell, q) ? d : -CUDART_INF_F;
        m = fmaxf(m, s[q]);
    }
    float Z = 0.f;
    o = zero_row<CE>();
#pragma unroll
    for (int q = 0; q < W; ++q) {
        s[q] = ex2_approx(s[q] - m);   // w_q
        Z += s[q];
#pragma unroll
        for (int c = 0; c < CE; ++c) o.v[c] = fmaf(s[q], xj[q].v[c], o.v[c]);
    }
    const float rZ = any ? rcp_refined(Z) : 0.f;
#pragma unroll
    for (int c = 0; c < CE; ++c) o.v[c] *= rZ;
    D = dot<CE>(go, o);
    lse = any ? m + lg2_approx(Z) : 0.f;   // empty row: never read by a source pass
    const float scale = rZ * LN2_F;
    t = zero_row<CE>();
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const float ds = (s[q] * scale) * (dot<CE>(go, xj[q]) - D);
#pragma unroll
        for (int c = 0; c < CE; ++c) t.v[c] = fmaf(ds, xj[q].v[c], t.v[c]);
    }
}

// ---- last forward layer fused with the destination pass of its backward ------------------------
// One gather of the row serves both.  p = project(Mu, y) comes from the caller (which can store it
// before the gathers: fewer live registers).  k = F(y) as ell_feval; gp = cot(k) = dL/dx^L at this node (the
// caller's node-local loss cotangent of x^L = y + b k); then, with go = b * gp, the outputs of ell_bwd_dst
// at xi = y from the same registers (w_q, m, Z, rZ).  Every term is ell_feval's / ell_bwd_dst's
// expression, so the bits equal those of the two separate passes.
template <int CE, int W, typename Cot>
__device__ __forceinline__ void ell_feval_bwd_dst(const unsigned char* __restrict__ Xb, const uint4& ell,
                                                  const Row<CE>& y, const Row<CE>& p, float b, Cot cot, Row<CE>& gp,
                                                  float& D, float& lse, Row<CE>& t, Row<CE>& o) {
    const bool any = ell_valid(ell) != 0;
    Row<CE> xj[W];
    float s[W];
    float m = -3.0e38f;
#pragma unroll
    for (int q = 0; q < W; ++q) {
        xj[q] = lds_row<CE>(Xb, ell_off(ell, q));
        const float d = dot<CE>(p, xj[q]);
        s[q] = ell_has(ell, q) ? d : -CUDART_INF_F;
        m = fmaxf(m, s[q]);
    }
    float Z = 0.f;
    o = zero_row<CE>();
#pragma unroll
    for (int q = 0; q < W; ++q) {
        s[q] = ex2_approx(s[q] - m);   // w_q
        Z += s[q];
#pragma unroll
        for (int c = 0; c < CE; ++c) o.v[c] = fmaf(s[q], xj[q].v[c], o.v[c]);
    }
    const float rZ = any ? rcp_refined(Z) : 0.f;
    Row<CE> k;
#pragma unroll
    for (int c = 0; c < CE; ++c) k.v[c] = fmaf(o.v[c], rZ, -y.v[c]);
    gp = cot(k);
    Row<CE> go;
#pragma unroll
    for (int c = 0; c < CE; ++c) go.v[c] = b * gp.v[c];
#pragma unroll
    for (int c = 0; c < CE; ++c) o.v[c] *= rZ;
    D = dot<CE>(go, o);
    lse = any ? m + lg2_approx(Z) : 0.f;
    const float scale = rZ * LN2_F;
    t = zero_row<CE>();
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const float ds = (s[q] * scale) * (dot<CE>(go, xj[q]) - D);
#pragma unroll
        for (int c = 0; c < CE; ++c) t.v[c] = fmaf(ds, xj[q].v[c], t.v[c]);
    }
}

// ---- backward, source pass ---------------------------------------------------------------------
// Contributions of the out-edges (j -> i) of node j:  sum_e alpha_e (go_i + c_e p_i),
// c_e = ln2 (<go_i, x_j> - D_i),  alpha_e = 2^(<p_i, x_j> - lse_i).
// Pb / Gb: rows p_i / go_i; DLb: float2 rows (D_i, lse_i), i.e. 8 bytes per node.
template <int CE, int W>
__device__ __forceinline__ Row<CE> ell_bwd_src(const unsigned char* __restrict__ Pb,
                                               const unsigned char* __restrict__ Gb,
                                               const unsigned char* __restrict__ DLb, const uint4& ell,
                                               const Row<CE>& xj) {
    Row<CE> acc = zero_row<CE>();
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const uint32_t off = ell_off(ell, q);
        const Row<CE> p = lds_row<CE>(Pb, off);
        const Row<CE> go = lds_row<CE>(Gb, off);
        const float2 dl = *reinterpret_cast<const float2*>(DLb + (CE == 4 ? (off >> 1) : off));
        const float sv = dot<CE>(p, xj) - dl.y;
        const float alpha = ex2_approx(ell_has(ell, q) ? sv : -CUDART_INF_F);
        const float c = (dot<CE>(go, xj) - dl.x) * LN2_F;
#pragma unroll
        for (int ch = 0; ch < CE; ++ch) acc.v[ch] = fmaf(alpha, fmaf(c, p.v[ch], go.v[ch]), acc.v[ch]);
    }
    return acc;
}

// ---- TMA bulk copy + mbarrier (sm_90+ PTX; SASS: UBLKCP / SYNCS) --------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 1-D bulk copy global -> shared; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    const uint32_t addr = smem_u32(bar);
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}

}  // namespace gad
