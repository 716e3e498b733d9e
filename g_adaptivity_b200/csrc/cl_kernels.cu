// Cluster-resident training kernel: one THREAD-BLOCK CLUSTER per mesh, for meshes too large for one
// CTA's shared memory (60x60 ... ~200x200 nodes) that the streaming kernels can only serve at L2
// speed.
//
// The mesh is cut into C contiguous slabs of nodes (C = cluster size, 2..16); CTA r of the cluster
// keeps slab r's state rows (X, X', P, GS, DL: 72 bytes per node) in its shared memory for the
// whole training pass, exactly like a tile of k_ell_train (ell_kernels.cuh).  A neighbour row that
// lives in another slab is read from that CTA's shared memory through distributed shared memory
// (mapa + ld.shared::cluster); the topology is a "cluster row" per node and direction,
//     crow[i] = { u32 e_0 .. e_6, u32 valid },   e_q = (owner rank << 24) | (row offset in bytes)
// streamed from L2 (32 bytes per node and pass).  Every phase boundary that another slab can see is a
// cluster barrier (barrier.cluster.arrive.release / wait.acquire) instead of __syncthreads().
//
// Same arithmetic as the mesh-resident kernels (ell_math.cuh), same per-CTA partial rows and the
// same tail (tail_prepare / tail_finish: reduction, chain rule, [peer all-reduce], Adam, refold) run
// by the last CTA to finish, so one training step is still ONE launch.
// Replaces src/run_GNN.py:99-131 (forward, mesh loss, backward, Adam) for such meshes.
#include <stdlib.h>

#include "ell_kernels.cuh"

namespace gad {
namespace cl {

using ell::Args;
using ell::Tracer;

constexpr int MAXT = 512;

struct CRow {
    uint32_t e[8];   // e[7] = validity mask
    __device__ __forceinline__ bool has(int q) const { return (e[7] >> q) & 1u; }
    __device__ __forceinline__ bool remote() const { return (e[7] >> 15) & 1u; }   // a neighbour lives in another slab
};

__device__ __forceinline__ CRow load_crow(const uint4* __restrict__ rows, int64_t i) {
    const uint4 a = __ldg(rows + 2 * i), b = __ldg(rows + 2 * i + 1);
    CRow r;
    r.e[0] = a.x; r.e[1] = a.y; r.e[2] = a.z; r.e[3] = a.w;
    r.e[4] = b.x; r.e[5] = b.y; r.e[6] = b.z; r.e[7] = b.w;
    return r;
}

__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_size() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
// Phase boundary of a cluster.  What has to cross it is SHARED memory only (every global value a
// thread reads back was written by itself): a CTA-scope fence orders this thread's shared-memory
// stores before its arrival, and a slab's rows are physically in its SM's shared memory by the time
// every thread of the cluster has arrived.  The default .release / .acquire forms would add a
// GPU-scope MEMBAR (waiting for the outstanding `states` stores to reach L2) and an L1 invalidation
// to each of the 13 barriers of a pass.  GAD_CLUSTER_STRICT_SYNC=1 at build time restores them.
__device__ __forceinline__ void cluster_sync() {
#if defined(GAD_CLUSTER_STRICT_SYNC) && GAD_CLUSTER_STRICT_SYNC
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
#else
    asm volatile("fence.acq_rel.cta;\n\tbarrier.cluster.arrive.relaxed.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
#endif
}

// row of CE floats at a shared::cluster address (own or a peer CTA's shared memory)
template <int CE>
__device__ __forceinline__ Row<CE> ldc_row(uint32_t caddr) {
    Row<CE> r;
    if constexpr (CE == 2) {
        asm volatile("ld.shared::cluster.v2.f32 {%0, %1}, [%2];" : "=f"(r.v[0]), "=f"(r.v[1]) : "r"(caddr) : "memory");
    } else {
        asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
                     : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3])
                     : "r"(caddr)
                     : "memory");
    }
    return r;
}
__device__ __forceinline__ float2 ldc_f2(uint32_t caddr) {
    float2 v;
    asm volatile("ld.shared::cluster.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(caddr) : "memory");
    return v;
}

struct Layout {
    uint32_t xa, xb, p, gs, dl, mu, red, bar, total;
};

__host__ __device__ inline Layout make_layout(int CE, int cap_nodes, int nwarps) {
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
    s.p = bump(rows);
    s.gs = bump(rows);
    s.dl = bump((size_t)cap_nodes * 8);
    s.mu = bump((size_t)(CE * CE + CE) * sizeof(float));
    s.red = bump((size_t)(CE * CE + CE + 1) * nwarps * sizeof(float));
    if (o < ell::TAIL_SCRATCH_MIN) o = ell::TAIL_SCRATCH_MIN;
    s.bar = bump(16);
    s.total = (uint32_t)o;
    return s;
}

// ---- backward of one slab (shared by the train and the backward kernels) ---------------------------------
// On entry: X = x^{L-1} rows of the slab (buffer at cluster offset offX), GS = dL/dx^L rows, Mu = weights of
// layer L-1 (with the bias offset of the mesh when DU: a.du, global CNN features); GO (offset offGO) is free.  Per-CTA
// partial rows go to a.partials[blockIdx.x].  DU is a template flag so that the kernels without the offset compile to
// what they were before it existed.
template <int CE, int W, bool DU>
__device__ __forceinline__ void cl_backward(const Args& a, const Layout& lay, int mesh, int n0, int NT, unsigned char* X,
                                            unsigned char* GO, uint32_t offX, uint32_t offGO, unsigned char* P,
                                            unsigned char* DL, unsigned char* GS, const uint4* __restrict__ Rin,
                                            const uint4* __restrict__ Rout, float* Mu, float* red,
                                            const uint32_t* __restrict__ s_base) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    constexpr int NACC = MUSZ + 1;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const size_t state_stride = (size_t)a.N * CE;
    const uint32_t offP = lay.p, offDL = lay.dl;
    const bool per_layer = (a.Lw > 1);
    const int slots = per_layer ? a.L : 1;
    float acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) acc[k] = 0.f;
    for (int l = a.L - 1; l >= 0; --l) {
        if (per_layer && l < a.L - 1) {
            if constexpr (DU) ell::load_mu<CE>(a, Mu, l, mesh);
            else for (int t = tid; t < MUSZ; t += nthr) Mu[t] = a.Mu[(size_t)l * MUSZ + t];
            __syncthreads();
        }
        const float b = __ldcg(a.tau + l);
        float gtau = 0.f;
        // phase A: destination pass (ell_math.cuh: ell_bwd_dst)
        for (int i = tid; i < NT; i += nthr) {
            const CRow e = load_crow(Rin, i);
            const Row<CE> xi = lds_row<CE>(X, i * RB);
            const Row<CE> gp = lds_row<CE>(GS, i * RB);
            Row<CE> go;
#pragma unroll
            for (int c = 0; c < CE; ++c) go.v[c] = b * gp.v[c];
            const bool any = (e.e[7] & 0x7fu) != 0;
            const Row<CE> p = project<CE>(Mu, xi);
            Row<CE> xj[W];
            float s[W];
            float m = -3.0e38f;
            if (__any_sync(__activemask(), e.remote())) {
#pragma unroll
                for (int q = 0; q < W; ++q) xj[q] = ldc_row<CE>(s_base[e.e[q] >> 24] + offX + (e.e[q] & 0xffffffu));
            } else {
#pragma unroll
                for (int q = 0; q < W; ++q) xj[q] = lds_row<CE>(X, e.e[q] & 0xffffffu);
            }
#pragma unroll
            for (int q = 0; q < W; ++q) {
                const float d = dot<CE>(p, xj[q]);
                s[q] = e.has(q) ? d : -CUDART_INF_F;
                m = fmaxf(m, s[q]);
            }
            float Z = 0.f;
            Row<CE> o = zero_row<CE>();
#pragma unroll
            for (int q = 0; q < W; ++q) {
                s[q] = ex2_approx(s[q] - m);
                Z += s[q];
#pragma unroll
                for (int c = 0; c < CE; ++c) o.v[c] = fmaf(s[q], xj[q].v[c], o.v[c]);
            }
            const float rZ = any ? rcp_refined(Z) : 0.f;
#pragma unroll
            for (int c = 0; c < CE; ++c) o.v[c] *= rZ;
            const float D = dot<CE>(go, o);
            const float lse = any ? m + lg2_approx(Z) : 0.f;
            const float scale = rZ * LN2_F;
            Row<CE> t = zero_row<CE>();
#pragma unroll
            for (int q = 0; q < W; ++q) {
                const float ds = (s[q] * scale) * (dot<CE>(go, xj[q]) - D);
#pragma unroll
                for (int c = 0; c < CE; ++c) t.v[c] = fmaf(ds, xj[q].v[c], t.v[c]);
            }
#pragma unroll
            for (int c = 0; c < CE; ++c) gtau = fmaf(gp.v[c], o.v[c] - xi.v[c], gtau);
#pragma unroll
            for (int aa = 0; aa < CE; ++aa)
#pragma unroll
                for (int bb = 0; bb < CE; ++bb) acc[aa * CE + bb] = fmaf(xi.v[aa], t.v[bb], acc[aa * CE + bb]);
#pragma unroll
            for (int bb = 0; bb < CE; ++bb) acc[CE * CE + bb] += t.v[bb];
            const Row<CE> Mt = apply_M<CE>(Mu, t);
            Row<CE> gs;
#pragma unroll
            for (int c = 0; c < CE; ++c) gs.v[c] = fmaf(1.0f - b, gp.v[c], Mt.v[c]);
            sts_row<CE>(P, i * RB, p);
            *reinterpret_cast<float2*>(DL + (size_t)i * 8) = make_float2(D, lse);
            sts_row<CE>(GO, i * RB, go);
            sts_row<CE>(GS, i * RB, gs);
        }
        if (l > 0 || a.g_x0) {
            cluster_sync();   // P, DL, GO of every slab visible; every gather of X done
            // phase B: source pass (ell_math.cuh: ell_bwd_src), then X <- x^{l-1}
            const float* xprev_g = (l > 0) ? a.states + (size_t)(l - 1) * state_stride : nullptr;
            for (int j = tid; j < NT; j += nthr) {
                const CRow e = load_crow(Rout, j);
                Row<CE> xprev = zero_row<CE>();
                if (xprev_g) xprev = ell::load_row_cg<CE>(xprev_g, (int64_t)n0 + j);
                const Row<CE> xj = lds_row<CE>(X, j * RB);
                Row<CE> g = lds_row<CE>(GS, j * RB);
                const bool warp_remote = __any_sync(__activemask(), e.remote());
#pragma unroll
                for (int q = 0; q < W; ++q) {
                    const uint32_t off = e.e[q] & 0xffffffu;
                    Row<CE> p, go;
                    float2 dl;
                    if (warp_remote) {
                        const uint32_t base = s_base[e.e[q] >> 24];
                        p = ldc_row<CE>(base + offP + off);
                        go = ldc_row<CE>(base + offGO + off);
                        dl = ldc_f2(base + offDL + (CE == 4 ? (off >> 1) : off));
                    } else {
                        p = lds_row<CE>(P, off);
                        go = lds_row<CE>(GO, off);
                        dl = *reinterpret_cast<const float2*>(DL + (CE == 4 ? (off >> 1) : off));
                    }
                    const float sv = dot<CE>(p, xj) - dl.y;
                    const float alpha = ex2_approx(e.has(q) ? sv : -CUDART_INF_F);
                    const float c = (dot<CE>(go, xj) - dl.x) * LN2_F;
#pragma unroll
                    for (int ch = 0; ch < CE; ++ch) g.v[ch] = fmaf(alpha, fmaf(c, p.v[ch], go.v[ch]), g.v[ch]);
                }
                sts_row<CE>(GS, j * RB, g);
                if (xprev_g) sts_row<CE>(X, j * RB, xprev);
                else store_row<CE>(a.g_x0, (int64_t)n0 + j, g);
            }
            cluster_sync();   // X of the next layer complete; gathers of P / DL / GO done
        }
        if (per_layer) {
            acc[NACC - 1] = gtau;
            block_reduce<NACC>(acc, red, a.partials + ((size_t)blockIdx.x * slots + l) * NACC);
#pragma unroll
            for (int k = 0; k < NACC; ++k) acc[k] = 0.f;
        } else if (a.tau_partials) {
            float one[1] = {gtau};
            block_reduce<1>(one, red, a.tau_partials + (size_t)blockIdx.x * a.L + l);
        }
    }
    if (!per_layer) block_reduce<NACC>(acc, red, a.partials + (size_t)blockIdx.x * NACC);
}

// a.tile_ptr = mesh_ptr [M + 1]; a.T = number of per-CTA partial rows (= grid); a.cap_nodes = slab capacity;
// a.ell_in / a.ell_out = cluster rows (2 x uint4 per node).  COT: loss_kind 2, the target rows hold the caller's
// cotangent of x_phys (ell_kernels.cuh: k_ell_train).
template <int CE, int W, bool COT = false>
__global__ void __launch_bounds__(MAXT, 1) k_cl_train(const Args a) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const Layout lay = make_layout(CE, a.cap_nodes, (nthr + 31) >> 5);
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
    __shared__ uint32_t s_base[16];   // shared::cluster address of every rank's dynamic shared memory
    ell::pdl_launch_dependents();
    Tracer tr{a.trace ? a.trace + (size_t)blockIdx.x * 64 : nullptr, 0};
    tr.mark();
    const uint32_t C = cluster_size(), rank = cluster_rank();
    const int mesh = (int)(blockIdx.x / C);
    const int m0 = a.tile_ptr[mesh], NM = a.tile_ptr[mesh + 1] - m0;
    const int S = ((NM + (int)C - 1) / (int)C + 3) & ~3;                  // slab size (multiple of 4 nodes)
    const int n0 = m0 + (int)rank * S;                                     // first node of this slab
    const int NT = max(0, min(S, NM - (int)rank * S));                     // nodes of this slab
    if (tid < 16) s_base[tid] = (tid < (int)C) ? mapa(smem_u32(smem), (uint32_t)tid) : 0u;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    const size_t state_stride = (size_t)a.N * CE;
    const uint4* Rin = a.ell_in + 2 * (size_t)n0;
    const uint4* Rout = a.ell_out + 2 * (size_t)n0;

    // ---- inputs of the slab by TMA bulk copies, features assembled before the wait on the previous step
    const uint32_t xc_bytes = (uint32_t)NT * (uint32_t)a.dim * 4u, sc_bytes = (uint32_t)NT * 4u;
    const float* xc_g = a.x_comp + (size_t)n0 * a.dim;
    const float* tg_g = a.target + (size_t)n0 * a.dim;
    const float* f_g = a.f ? a.f + n0 : nullptr;
    const float* uu_g = a.uu ? a.uu + n0 : nullptr;
    const bool stage = NT > 0 && a.dim <= 2 && (NT % 4 == 0) && (xc_bytes % 16 == 0) &&
                       ((reinterpret_cast<uintptr_t>(xc_g) | reinterpret_cast<uintptr_t>(tg_g) |
                         reinterpret_cast<uintptr_t>(f_g) | reinterpret_cast<uintptr_t>(uu_g)) & 15) == 0;
    unsigned char* st_xc = P;
    unsigned char* st_f = P + xc_bytes;
    unsigned char* st_uu = st_f + (a.f ? sc_bytes : 0u);
    const uint32_t tx = stage ? 2u * xc_bytes + (a.f ? sc_bytes : 0u) + (a.uu ? sc_bytes : 0u) : 0u;
    if (tid == 0 && tx) {
        fence_proxy_async_smem();
        mbar_expect_tx(bar, tx);
        bulk_g2s(st_xc, xc_g, xc_bytes, bar);
        if (a.f) bulk_g2s(st_f, f_g, sc_bytes, bar);
        if (a.uu) bulk_g2s(st_uu, uu_g, sc_bytes, bar);
        bulk_g2s(DL, tg_g, xc_bytes, bar);
    }
    if (tx) mbar_wait(bar, 0);
    unsigned char* Xc = B0;
    unsigned char* Xn = B1;
    ell::assemble_rows<CE>(a, n0, NT, stage, st_xc, st_f, st_uu, Xc, nullptr);
    ell::pdl_wait();
    if (a.tail >= 2 && tid == nthr - 1) {
        s_step = __ldcg(a.step) + 1;
        s_coef = tail::adam_coef(a.lr, a.beta1, a.beta2, a.eps, a.weight_decay, a.adam_grad_scale, s_step);
    }
    for (int t = tid; t < MUSZ; t += nthr) Mu[t] = __ldcg(a.Mu + t);
    cluster_sync();   // every slab's x^0 is in place (and Mu / s_base visible to the block)
    tr.mark();

    const uint32_t offXc0 = lay.xa, offXn0 = lay.xb;
    uint32_t offXc = offXc0, offXn = offXn0;

    // ---- forward (Euler), loss and cotangent fused into the last layer ----------------------------
    float loss_acc = 0.f;
    for (int l = 0; l < a.L; ++l) {
        if (a.Lw > 1 && l > 0) {
            for (int t = tid; t < MUSZ; t += nthr) Mu[t] = a.Mu[(size_t)l * MUSZ + t];
            __syncthreads();
        }
        const float h = __ldcg(a.tau + l);
        const bool last = (l == a.L - 1);
        float* st_out = last ? nullptr : a.states + (size_t)(l + 1) * state_stride;
        float Mr[MUSZ];
#pragma unroll
        for (int t = 0; t < MUSZ; ++t) Mr[t] = Mu[t];
        for (int i = tid; i < NT; i += nthr) {
            const CRow e = load_crow(Rin, i);
            const Row<CE> y = lds_row<CE>(Xc, i * RB);
            if (l == 0) store_row<CE>(a.states, (int64_t)n0 + i, y);
            // F(y) at node i (ell_math.cuh: ell_feval), neighbour rows through shared::cluster addresses
            const bool any = (e.e[7] & 0x7fu) != 0;
            const Row<CE> p = project<CE>(Mr, y);
            Row<CE> xj[W];
            float s[W];
            float m = -3.0e38f;
            if (__any_sync(__activemask(), e.remote())) {   // some row of this warp lives in another slab
#pragma unroll
                for (int q = 0; q < W; ++q) xj[q] = ldc_row<CE>(s_base[e.e[q] >> 24] + offXc + (e.e[q] & 0xffffffu));
            } else {                                        // interior warp: plain shared-memory loads
#pragma unroll
                for (int q = 0; q < W; ++q) xj[q] = lds_row<CE>(Xc, e.e[q] & 0xffffffu);
            }
#pragma unroll
            for (int q = 0; q < W; ++q) {
                const float d = dot<CE>(p, xj[q]);
                s[q] = e.has(q) ? d : -CUDART_INF_F;
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
            const float rZ = any ? rcp_refined(Z) : 0.f;
            Row<CE> xn;
#pragma unroll
            for (int c = 0; c < CE; ++c) xn.v[c] = fmaf(h, fmaf(o.v[c], rZ, -y.v[c]), y.v[c]);
            if (!last) {
                sts_row<CE>(Xn, i * RB, xn);
                store_row<CE>(st_out, (int64_t)n0 + i, xn);
            } else {
                const int64_t gi = (int64_t)n0 + i;
                if (a.x_phys) ell::store_dims<CE>(a.x_phys, gi, a.dim, xn);
                const Row<CE> tg = stage ? ell::load_dims<CE>(reinterpret_cast<const float*>(DL), i, a.dim)
                                         : ell::load_dims<CE>(a.target, gi, a.dim);
                Row<CE> g;
#pragma unroll
                for (int c = 0; c < CE; ++c) {
                    if constexpr (COT) {
                        const float cc = (c < a.dim) ? tg.v[c] : 0.f;
                        loss_acc = fmaf(xn.v[c], cc, loss_acc);
                        g.v[c] = a.grad_scale * cc;
                    } else {
                        const float d = (c < a.dim) ? xn.v[c] - tg.v[c] : 0.f;
                        if (a.loss_kind == 0) {
                            loss_acc += fabsf(d);
                            g.v[c] = (d > 0.f) ? a.grad_scale : ((d < 0.f) ? -a.grad_scale : 0.f);
                        } else {
                            loss_acc = fmaf(d, d, loss_acc);
                            g.v[c] = 2.0f * a.grad_scale * d;
                        }
                    }
                }
                sts_row<CE>(GS, i * RB, g);
            }
        }
        cluster_sync();   // x^{l+1} of every slab complete; all gathers of x^l done
        if (!last) {
            unsigned char* t = Xc; Xc = Xn; Xn = t;
            const uint32_t u = offXc; offXc = offXn; offXn = u;
        }
    }
    {
        float one[1] = {loss_acc};
        block_reduce<1>(one, red, a.loss_partials + blockIdx.x);
    }
    tr.mark();

    // ---- backward: Xc = x^{L-1}, Xn = free -> GO ---------------------------------------------------
    cl_backward<CE, W, false>(a, lay, mesh, n0, NT, Xc, Xn, offXc, offXn, P, DL, GS, Rin, Rout, Mu, red, s_base);
    tr.mark();
    // no CTA may leave while a peer can still read its shared memory
    cluster_sync();

    // ---- tail: the last CTA of the GRID to finish (ell_kernels.cuh) ---------------------------------
    if (a.tail == 0) return;
    if (tid < 32) {
        __threadfence();
        __syncwarp();
        if (tid == 0) {
            const unsigned int prev = atomicAdd(a.counter, 1u);
            s_last = (prev == gridDim.x - 1) ? 1 : 0;
        }
    }
    __syncthreads();
    if (!s_last) return;
    ell::TailCtx cx;
    ell::tail_prepare<CE>(a, smem, lay.bar, cx);
    __threadfence();
    ell::tail_finish<CE>(a, smem, cx, s_coef, s_step, tr);
    if (tid == 0) *a.counter = 0u;
}

// ---- backward only (autograd of the module seam): from the saved layer inputs ---------------------------
// DU: a.du holds the per-mesh bias offset (global CNN features)
template <int CE, int W, bool DU>
__global__ void __launch_bounds__(MAXT, 1) k_cl_bwd(const Args a) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const Layout lay = make_layout(CE, a.cap_nodes, (nthr + 31) >> 5);
    unsigned char* X = smem + lay.xa;
    unsigned char* GO = smem + lay.xb;
    unsigned char* P = smem + lay.p;
    unsigned char* GS = smem + lay.gs;
    unsigned char* DL = smem + lay.dl;
    float* Mu = reinterpret_cast<float*>(smem + lay.mu);
    float* red = reinterpret_cast<float*>(smem + lay.red);
    __shared__ uint32_t s_base[16];
    const uint32_t C = cluster_size(), rank = cluster_rank();
    const int mesh = (int)(blockIdx.x / C);
    const int m0 = a.tile_ptr[mesh], NM = a.tile_ptr[mesh + 1] - m0;
    const int S = ((NM + (int)C - 1) / (int)C + 3) & ~3;
    const int n0 = m0 + (int)rank * S;
    const int NT = max(0, min(S, NM - (int)rank * S));
    if (tid < 16) s_base[tid] = (tid < (int)C) ? mapa(smem_u32(smem), (uint32_t)tid) : 0u;
    const size_t state_stride = (size_t)a.N * CE;
    const float* xl = a.states + (size_t)(a.L - 1) * state_stride;
    for (int i = tid; i < NT; i += nthr) {
        sts_row<CE>(X, i * RB, ell::load_row_cg<CE>(xl, (int64_t)n0 + i));
        sts_row<CE>(GS, i * RB, ell::load_dims<CE>(a.g_xphys, (int64_t)n0 + i, a.dim));   // cotangent of x^L[:, :dim]
    }
    const int lw = (a.Lw > 1) ? a.L - 1 : 0;
    if constexpr (DU) ell::load_mu<CE>(a, Mu, lw, mesh);
    else for (int t = tid; t < MUSZ; t += nthr) Mu[t] = a.Mu[(size_t)lw * MUSZ + t];
    cluster_sync();
    cl_backward<CE, W, DU>(a, lay, mesh, n0, NT, X, GO, lay.xa, lay.xb, P, DL, GS, a.ell_in + 2 * (size_t)n0,
                       a.ell_out + 2 * (size_t)n0, Mu, red, s_base);
    cluster_sync();   // nobody leaves while a peer may still read its shared memory
}

// fixed-order fp64 sums of the per-CTA partial rows: one warp per output column (ell_api.cu: k_ell_reduce)
__global__ void k_cl_reduce(const float* __restrict__ partials, int T, int slots, int nacc, int musz, float* __restrict__ gMu,
                            const float* __restrict__ tau_partials, int L, float* __restrict__ g_tau) {
    tail::reduce_partials(partials, T, slots, nacc, musz, gMu, tau_partials, L, g_tau, nullptr, 0.f, nullptr,
                          blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), gridDim.x * (blockDim.x >> 5));
}

// d loss / d du [M, Lw, CE] (global CNN features): G_u of the cluster's C per-CTA partial rows, summed in rank order
__global__ void k_cl_du_reduce(const float* __restrict__ partials, int M, int C, int Lw, int slots, int nacc, int CE,
                               float* __restrict__ g_du) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= M * Lw * CE) return;
    const int z = k % CE, lw = (k / CE) % Lw, b = k / (CE * Lw);
    const int slot = (slots > 1) ? lw : 0;
    double s = 0.0;
    for (int r = 0; r < C; ++r) s += (double)partials[((size_t)(b * C + r) * slots + slot) * nacc + CE * CE + z];
    g_du[k] = (float)s;
}

// ---- forward only (module seam / inference): Euler layers or classical RK4 steps -------------------------
// F(y) = A(y) y - y at node i of this slab, neighbour rows of the state buffer at `offX`
template <int CE, int W>
__device__ __forceinline__ Row<CE> cl_feval(const CRow& e, const Row<CE>& y, const float* __restrict__ Mu,
                                            const unsigned char* __restrict__ Xloc, uint32_t offX,
                                            const uint32_t* __restrict__ s_base) {
    const bool any = (e.e[7] & 0x7fu) != 0;
    const Row<CE> p = project<CE>(Mu, y);
    Row<CE> xj[W];
    float s[W];
    float m = -3.0e38f;
    if (__any_sync(__activemask(), e.remote())) {
#pragma unroll
        for (int q = 0; q < W; ++q) xj[q] = ldc_row<CE>(s_base[e.e[q] >> 24] + offX + (e.e[q] & 0xffffffu));
    } else {
#pragma unroll
        for (int q = 0; q < W; ++q) xj[q] = lds_row<CE>(Xloc, e.e[q] & 0xffffffu);
    }
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const float d = dot<CE>(p, xj[q]);
        s[q] = e.has(q) ? d : -CUDART_INF_F;
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
    const float rZ = any ? rcp_refined(Z) : 0.f;
    Row<CE> k;
#pragma unroll
    for (int c = 0; c < CE; ++c) k.v[c] = fmaf(o.v[c], rZ, -y.v[c]);
    return k;
}

// One cluster per mesh, the state resident in shared memory for ALL layers / RK4 steps of the call
// (BASELINE config 4: a 200x200 mesh, 64 RK4 steps = 256 F-evaluations, is one launch of 16 CTAs
// instead of 256 dependent launches).  Inputs are the raw features (src/GNN.py:225-239).
template <int CE, int W, int METHOD, bool DU>
__global__ void __launch_bounds__(MAXT, 1) k_cl_fwd(const Args a) {
    constexpr uint32_t RB = CE * sizeof(float);
    constexpr int MUSZ = CE * CE + CE;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const Layout lay = make_layout(CE, a.cap_nodes, (nthr + 31) >> 5);
    unsigned char* Xc = smem + lay.xa;
    unsigned char* Xn = smem + lay.xb;
    unsigned char* XB = smem + lay.p;    // RK4: the step's base state
    unsigned char* AC = smem + lay.gs;   // RK4: k1 + 2 k2 + 2 k3
    float* Mu = reinterpret_cast<float*>(smem + lay.mu);
    __shared__ uint32_t s_base[16];
    const uint32_t C = cluster_size(), rank = cluster_rank();
    const int mesh = (int)(blockIdx.x / C);
    const int m0 = a.tile_ptr[mesh], NM = a.tile_ptr[mesh + 1] - m0;
    const int S = ((NM + (int)C - 1) / (int)C + 3) & ~3;
    const int n0 = m0 + (int)rank * S;
    const int NT = max(0, min(S, NM - (int)rank * S));
    if (tid < 16) s_base[tid] = (tid < (int)C) ? mapa(smem_u32(smem), (uint32_t)tid) : 0u;
    if constexpr (DU) ell::load_mu<CE>(a, Mu, 0, mesh);
    else for (int t = tid; t < MUSZ; t += nthr) Mu[t] = a.Mu[t];
    const size_t state_stride = (size_t)a.N * CE;
    const uint4* Rin = a.ell_in + 2 * (size_t)n0;
    ell::assemble_rows<CE>(a, n0, NT, false, nullptr, nullptr, nullptr, Xc, a.states);
    cluster_sync();
    uint32_t offXc = lay.xa, offXn = lay.xb;
    for (int l = 0; l < a.L; ++l) {
        if (a.Lw > 1 && l > 0) {
            __syncthreads();
            if constexpr (DU) ell::load_mu<CE>(a, Mu, l, mesh);
            else for (int t = tid; t < MUSZ; t += nthr) Mu[t] = a.Mu[(size_t)l * MUSZ + t];
            __syncthreads();
        }
        const float h = a.tau[l];
        const bool last = (l == a.L - 1);
        float* st_out = (a.states && !last) ? a.states + (size_t)(l + 1) * state_stride : nullptr;
        if constexpr (METHOD == GAD_METHOD_EULER) {
            for (int i = tid; i < NT; i += nthr) {
                const CRow e = load_crow(Rin, i);
                const Row<CE> y = lds_row<CE>(Xc, i * RB);
                const Row<CE> k = cl_feval<CE, W>(e, y, Mu, Xc, offXc, s_base);
                Row<CE> xn;
#pragma unroll
                for (int c = 0; c < CE; ++c) xn.v[c] = fmaf(h, k.v[c], y.v[c]);
                sts_row<CE>(Xn, i * RB, xn);
                if (st_out) store_row<CE>(st_out, (int64_t)n0 + i, xn);
                if (last) ell::store_dims<CE>(a.x_phys, (int64_t)n0 + i, a.dim, xn);
            }
            cluster_sync();
            unsigned char* t = Xc; Xc = Xn; Xn = t;
            const uint32_t u = offXc; offXc = offXn; offXn = u;
        } else {
            // classical RK4 on F (extension, SURVEY A.1; same staging as ell_kernels.cuh: k_ell_fwd)
            const float cin[4] = {0.5f * h, 0.5f * h, h, 0.f};
            const float wacc[4] = {1.f, 2.f, 2.f, 1.f};
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                for (int i = tid; i < NT; i += nthr) {
                    const CRow e = load_crow(Rin, i);
                    const Row<CE> y = lds_row<CE>(Xc, i * RB);
                    const Row<CE> k = cl_feval<CE, W>(e, y, Mu, Xc, offXc, s_base);
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
                        if (last) ell::store_dims<CE>(a.x_phys, (int64_t)n0 + i, a.dim, out);
                    }
                    sts_row<CE>(Xn, i * RB, out);
                }
                cluster_sync();
                unsigned char* t = Xc; Xc = Xn; Xn = t;
                const uint32_t u = offXc; offXc = offXn; offXn = u;
            }
        }
    }
    cluster_sync();   // nobody leaves while a peer may still read its shared memory
}

// ---- cluster rows from the (row-sorted) CSR / CSC walk arrays -----------------------------------------
// grid.y = mesh; e_q = (rank << 24) | (row-in-slab * rowbytes); unused slots = the node itself, masked.
__global__ void __launch_bounds__(256) k_build_crows(const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                                                    const int32_t* __restrict__ mesh_ptr, int C, int rowbytes,
                                                    uint4* __restrict__ rows, int32_t* __restrict__ bad) {
    const int mesh = blockIdx.y;
    const int m0 = mesh_ptr[mesh], NM = mesh_ptr[mesh + 1] - m0;
    const int S = ((NM + C - 1) / C + 3) & ~3;
    for (int li = blockIdx.x * blockDim.x + threadIdx.x; li < NM; li += gridDim.x * blockDim.x) {
        const int i = m0 + li;
        const int b = ptr[i], deg = ptr[i + 1] - b;
        uint32_t v[8];
        bool ok = deg <= 7, remote = false;
#pragma unroll
        for (int q = 0; q < 7; ++q) {
            int j = (ok && q < deg) ? idx[b + q] : i;
            if (j < m0 || j >= m0 + NM) {
                ok = false;
                j = i;
            }
            const int lj = j - m0, r = lj / S;
            v[q] = ((uint32_t)r << 24) | (uint32_t)((lj - r * S) * rowbytes);
            remote |= (r != li / S);
        }
        v[7] = ok ? (((deg >= 7) ? 0x7fu : ((1u << deg) - 1u)) | (remote ? 0x8000u : 0u)) : 0u;
        if (!ok) atomicAdd(bad, 1);
        rows[2 * (size_t)i] = make_uint4(v[0], v[1], v[2], v[3]);
        rows[2 * (size_t)i + 1] = make_uint4(v[4], v[5], v[6], v[7]);
    }
}

int slots_for(int max_deg) { return max_deg <= 2 ? 2 : (max_deg <= 3 ? 3 : (max_deg <= 6 ? 6 : 7)); }

// slab capacity (nodes) one CTA can hold
int slab_cap(int CE) {
    const size_t fixed = 4096;   // Mu, red, bar, static shared memory, alignment
    const size_t avail = (size_t)smem_optin_bytes() - fixed;
    return (int)(avail / (size_t)(4 * CE * 4 + 8)) & ~3;
}

template <int CE, int W>
int launch_t(const Args& a, int C, int grid, int threads, cudaStream_t st) {
    auto kern = a.loss_kind == 2 ? k_cl_train<CE, W, true> : k_cl_train<CE, W, false>;
    const size_t bytes = make_layout(CE, a.cap_nodes, (threads + 31) / 32).total;
    GAD_CHECK_ARG((int)bytes <= smem_optin_bytes(), "cluster kernel: slab of %d nodes needs %zu B of shared memory",
                  a.cap_nodes, bytes);
    GAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    if (C > 8) GAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    int na = 1;
    if (a.pdl) {
        attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[1].val.programmaticStreamSerializationAllowed = 1;
        na = 2;
    }
    cfg.attrs = attr;
    cfg.numAttrs = na;
    GAD_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    count_launch(1);
    return GAD_OK;
}

}  // namespace cl
}  // namespace gad

using namespace gad;

extern "C" int gad_cluster_plan(int CE, int max_mesh_nodes, int max_cluster, int* cluster_size, int* slab_nodes) {
    GAD_CHECK_ARG((CE == 2 || CE == 4) && max_mesh_nodes > 0 && cluster_size && slab_nodes, "gad_cluster_plan: bad arguments");
    const int cap = cl::slab_cap(CE);
    // Measured on B200 (64 x 100x100 meshes): clusters of 4 run 146 us/step, of 8 253 us, of 16 217 us
    // against 204 us on the streaming kernels -- GPC packing and barrier cost grow with the cluster --
    // so the plan stops at 4 slabs (meshes up to ~12.6 k nodes) unless GAD_CLUSTER_MAX says otherwise.
    const int cmin = getenv("GAD_CLUSTER_MIN") ? atoi(getenv("GAD_CLUSTER_MIN")) : 2;
    // (max_cluster <= 0: that default; the forward-only kernel of a single large mesh takes up to 16)
    const int cmax = getenv("GAD_CLUSTER_MAX") ? atoi(getenv("GAD_CLUSTER_MAX")) : (max_cluster > 0 ? max_cluster : 4);
    for (int C = 2; C <= 16 && C <= cmax; C *= 2) {
        if (C < cmin) continue;
        const int S = ((max_mesh_nodes + C - 1) / C + 3) & ~3;
        if (S <= cap && (long long)S * CE * 4 < (1 << 24)) {
            *cluster_size = C;
            *slab_nodes = S;
            return GAD_OK;
        }
    }
    set_error("gad_cluster_plan: a mesh of %d nodes does not fit %d slabs of %d nodes", max_mesh_nodes, cmax, cap);
    return GAD_ERR_UNSUPPORTED;
}

extern "C" int gad_graph_build_cluster(const int32_t* ptr, const int32_t* idx, const int32_t* mesh_ptr, int M,
                                       int max_mesh_nodes, int CE, int cluster_size, void* rows, int32_t* info,
                                       void* stream) {
    GAD_CHECK_ARG(ptr && idx && mesh_ptr && rows && info && M > 0 && max_mesh_nodes > 0, "gad_graph_build_cluster: bad arguments");
    GAD_CHECK_ARG((CE == 2 || CE == 4) && cluster_size >= 1 && cluster_size <= 16, "gad_graph_build_cluster: CE=%d C=%d", CE,
                  cluster_size);
    dim3 grid((unsigned)((max_mesh_nodes + 255) / 256), (unsigned)M);
    cl::k_build_crows<<<grid, 256, 0, as_stream(stream)>>>(ptr, idx, mesh_ptr, cluster_size, CE * 4,
                                                           reinterpret_cast<uint4*>(rows), info + GAD_INFO_ELL_BAD);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

/* How many clusters of `cluster_size` CTAs (slabs of `slab_nodes`) the device can hold at once. */
extern "C" int gad_cluster_occupancy(int CE, int cluster_size, int slab_nodes, int threads, int* max_active_clusters) {
    GAD_CHECK_ARG((CE == 2 || CE == 4) && max_active_clusters, "gad_cluster_occupancy: bad arguments");
    const size_t bytes = cl::make_layout(CE, slab_nodes, (threads + 31) / 32).total;
    auto kernel = (CE == 4) ? (const void*)cl::k_cl_train<4, 6> : (const void*)cl::k_cl_train<2, 2>;
    GAD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    if (cluster_size > 8) GAD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)cluster_size * 64);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = bytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cluster_size;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    GAD_CUDA(cudaOccupancyMaxActiveClusters(max_active_clusters, kernel, &cfg));
    return GAD_OK;
}

extern "C" size_t gad_cluster_workspace_bytes(int CE, int M, int cluster_size, int L) {
    return gad_ell_workspace_bytes(CE, M * cluster_size, L);
}

/* One whole training step on cluster-resident meshes: gad_train_step_ell's contract with
 * ell_in / ell_out = cluster rows (gad_graph_build_cluster), tile_ptr = mesh_ptr [T + 1], T = meshes,
 * max_tile_nodes = largest mesh. */
extern "C" int gad_train_step_cluster(const gad_train_desc* d, int cluster_size, void* stream) {
    GAD_CHECK_ARG(d, "gad_train_step_cluster: null descriptor");
    GAD_CHECK_ARG(d->ell_in && d->ell_out && d->tile_ptr && d->x_comp && d->target && d->Mu && d->tau && d->states &&
                      d->gMu && d->loss && d->workspace && d->counter,
                  "gad_train_step_cluster: null pointer");
    GAD_CHECK_ARG(d->N > 0 && d->T > 0 && d->L > 0 && d->dim >= 1 && d->dim <= d->CE && (d->Lw == 1 || d->Lw == d->L) &&
                      (d->CE == 2 || d->CE == 4),
                  "gad_train_step_cluster: N=%lld T=%d L=%d dim=%d CE=%d Lw=%d", (long long)d->N, d->T, d->L, d->dim, d->CE,
                  d->Lw);
    GAD_CHECK_ARG(d->dim + (d->f ? 1 : 0) + (d->uu ? 1 : 0) <= d->CE, "gad_train_step_cluster: input features exceed CE=%d",
                  d->CE);
    GAD_CHECK_ARG(d->loss_kind >= 0 && d->loss_kind <= 2, "gad_train_step_cluster: unknown loss kind %d", d->loss_kind);
    GAD_CHECK_ARG(d->tail == 1 || d->tail == 2, "gad_train_step_cluster: tail must be 1 or 2");
    GAD_CHECK_ARG(d->Wq && d->bq && d->Wk && d->gWq && d->gbq && d->gWk && d->gbk && d->C > 0,
                  "gad_train_step_cluster: the tail needs the Linear parameters and their gradient buffers");
    GAD_CHECK_ARG(d->tail < 2 || (d->params && d->grads && d->exp_avg && d->exp_avg_sq && d->step && d->n_params > 0),
                  "gad_train_step_cluster: tail == 2 needs the flat parameter vector and the Adam state");
    const int C = cluster_size;
    GAD_CHECK_ARG(C >= 2 && C <= 16 && (C & (C - 1)) == 0, "gad_train_step_cluster: cluster size %d", C);
    const int S = ((d->max_tile_nodes + C - 1) / C + 3) & ~3;
    const int grid = d->T * C;
    GAD_CHECK_ARG(d->workspace_bytes >= gad_ell_workspace_bytes(d->CE, grid, d->L), "gad_train_step_cluster: workspace too small");
    int threads = ((S + 3) / 4 + 31) / 32 * 32;   // about four rounds of nodes per thread
    if (threads < 128) threads = 128;
    if (threads > cl::MAXT) threads = cl::MAXT;
    // two slabs per SM when their shared memory allows it: 256 threads x 125 registers each
    if (2 * (cl::make_layout(d->CE, S, 8).total + 1024) <= 233472 && threads > 256) threads = 256;
    if (getenv("GAD_CLUSTER_THREADS")) threads = atoi(getenv("GAD_CLUSTER_THREADS"));
    const int NACC = d->CE * d->CE + d->CE + 1;
    float* ws = reinterpret_cast<float*>(d->workspace);
    ell::Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(d->ell_in);
    a.ell_out = reinterpret_cast<const uint4*>(d->ell_out);
    a.tile_ptr = d->tile_ptr;
    a.T = grid;
    a.cap_nodes = S;
    a.N = d->N;
    a.Mu = d->Mu;
    a.tau = d->tau;
    a.Lw = d->Lw;
    a.L = d->L;
    a.dim = d->dim;
    a.x_phys = d->x_phys;
    a.states = d->states;
    a.partials = ws;
    a.tau_partials = (d->g_tau && d->Lw == 1) ? ws + (size_t)grid * d->L * NACC : nullptr;
    a.x_comp = d->x_comp;
    a.f = d->f;
    a.uu = d->uu;
    a.f_scale = d->f_scale;
    a.uu_scale = d->uu_scale;
    a.target = d->target;
    a.loss_kind = d->loss_kind;
    a.grad_scale = d->grad_scale;
    a.loss_partials = ws + (size_t)grid * d->L * NACC + (size_t)grid * d->L;
    a.tail = d->tail;
    a.counter = d->counter;
    a.gMu = d->gMu;
    a.g_tau = d->g_tau;
    a.loss = d->loss;
    a.loss_scale = d->loss_scale;
    a.Wq = d->Wq;
    a.bq = d->bq;
    a.Wk = d->Wk;
    a.gWq = d->gWq;
    a.gbq = d->gbq;
    a.gWk = d->gWk;
    a.gbk = d->gbk;
    a.C = d->C;
    a.inv_temp = d->inv_temp;
    a.cfold = tail::fold_scale(d->inv_temp, d->C);
    a.Mu_next = d->Mu;
    a.params = d->params;
    a.grads = d->grads;
    a.exp_avg = d->exp_avg;
    a.exp_avg_sq = d->exp_avg_sq;
    a.n_params = d->n_params;
    a.lr = d->lr;
    a.beta1 = d->beta1;
    a.beta2 = d->beta2;
    a.eps = d->eps;
    a.weight_decay = d->weight_decay;
    a.adam_grad_scale = d->adam_grad_scale;
    a.step = reinterpret_cast<long long*>(d->step);
    a.pdl = (d->flags & GAD_TRAIN_PDL) ? 1 : 0;
    a.rank = d->rank;
    a.world = d->world;
    a.peers = d->peers;
    a.peer_seq = d->peer_seq;
    a.peer_timeout_ns = (unsigned long long)(d->peer_timeout_ms ? d->peer_timeout_ms : 10000u) * 1000000ull;
    a.trace = reinterpret_cast<long long*>(d->trace);
    // the in-kernel tail needs its scratch plan to fit and the flat-vector views (as gad_train_step_ell)
    const cl::Layout lay = cl::make_layout(d->CE, S, (threads + 31) / 32);
    const long long np = d->tail >= 2 ? d->n_params : 0;
    auto within = [](const float* q, const float* base, long long n) { return q >= base && q < base + n; };
    const ell::TailPlan tplan = ell::plan_tail(d->CE, d->Lw, d->L, d->C, a.tau_partials && a.g_tau, true, np, grid,
                                               (threads + 31) / 32, lay.bar);
    bool ok = tplan.ok;
    if (d->world > 1 && d->peers)   // received peer gradients [world][n_params] sit in the tail's staging area
        ok = ok && d->peer_seq && (size_t)d->world * (size_t)np * sizeof(float) <= tplan.stage_bytes;
    if (d->tail >= 2) {
        const float* views[] = {d->Wq, d->bq, d->Wk};
        const float* gviews[] = {d->gWq, d->gbq, d->gWk, d->gbk};
        for (const float* v : views) ok = ok && within(v, d->params, np);
        for (const float* v : gviews) ok = ok && within(v, d->grads, np);
        if (d->g_tau) ok = ok && within(d->g_tau, d->grads, np);
    }
    GAD_CHECK_ARG(ok, "gad_train_step_cluster: the in-kernel tail needs flat parameter / gradient views and %u B of scratch",
                  lay.bar);
    const int w = cl::slots_for(d->max_deg);
    cudaStream_t st = as_stream(stream);
    if (d->CE == 4 && w == 6) return cl::launch_t<4, 6>(a, C, grid, threads, st);
    if (d->CE == 4 && w == 7) return cl::launch_t<4, 7>(a, C, grid, threads, st);
    if (d->CE == 4) return cl::launch_t<4, 3>(a, C, grid, threads, st);
    if (w <= 2) return cl::launch_t<2, 2>(a, C, grid, threads, st);
    return cl::launch_t<2, 3>(a, C, grid, threads, st);
}

namespace gad {
namespace cl {
template <int CE, int W, int METHOD>
int launch_fwd_t(const Args& a, int C, int grid, int threads, cudaStream_t st) {
    auto kern = a.du ? k_cl_fwd<CE, W, METHOD, true> : k_cl_fwd<CE, W, METHOD, false>;
    const size_t bytes = make_layout(CE, a.cap_nodes, (threads + 31) / 32).total;
    GAD_CHECK_ARG((int)bytes <= smem_optin_bytes(), "cluster kernel: slab of %d nodes needs %zu B of shared memory",
                  a.cap_nodes, bytes);
    GAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    if (C > 8) GAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    GAD_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    count_launch(1);
    return GAD_OK;
}
}  // namespace cl
}  // namespace gad

/* Deformer forward from the raw inputs on cluster-resident meshes, ONE launch for all L layers / RK4
 * steps (gad_deform_fwd_ell_raw's contract with cluster rows, mesh_ptr [M + 1] and the cluster size;
 * du [M, Lw, CE] or NULL: per-mesh bias offset). */
extern "C" int gad_deform_fwd_cluster(const void* crows_in, const int32_t* mesh_ptr, int M, int max_mesh_nodes,
                                      int max_deg, int cluster_size, int64_t N, const float* x_comp, const float* f,
                                      const float* uu, const float* f_scale, const float* uu_scale, int dim, int CE,
                                      const float* Mu, const float* du, int Lw, const float* tau, int L, int method,
                                      float* x_phys, float* states, void* stream) {
    GAD_CHECK_ARG(crows_in && mesh_ptr && x_comp && Mu && tau && x_phys, "gad_deform_fwd_cluster: null pointer");
    GAD_CHECK_ARG(N > 0 && M > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L) && (CE == 2 || CE == 4),
                  "gad_deform_fwd_cluster: N=%lld M=%d L=%d dim=%d CE=%d Lw=%d", (long long)N, M, L, dim, CE, Lw);
    GAD_CHECK_ARG(dim + (f ? 1 : 0) + (uu ? 1 : 0) <= CE, "gad_deform_fwd_cluster: input features exceed CE=%d", CE);
    GAD_CHECK_ARG(method == GAD_METHOD_EULER || method == GAD_METHOD_RK4, "gad_deform_fwd_cluster: unknown method %d", method);
    const int C = cluster_size;
    GAD_CHECK_ARG(C >= 2 && C <= 16 && (C & (C - 1)) == 0, "gad_deform_fwd_cluster: cluster size %d", C);
    const int S = ((max_mesh_nodes + C - 1) / C + 3) & ~3;
    int threads = ((S + 3) / 4 + 31) / 32 * 32;
    if (threads < 128) threads = 128;
    if (threads > cl::MAXT) threads = cl::MAXT;
    ell::Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(crows_in);
    a.tile_ptr = mesh_ptr;
    a.T = M * C;
    a.cap_nodes = S;
    a.N = N;
    a.Mu = Mu;
    a.du = du;
    a.tau = tau;
    a.Lw = Lw;
    a.L = L;
    a.dim = dim;
    a.x_comp = x_comp;
    a.f = f;
    a.uu = uu;
    a.f_scale = f_scale;
    a.uu_scale = uu_scale;
    a.x_phys = x_phys;
    a.states = states;
    const int w = cl::slots_for(max_deg);
    cudaStream_t st = as_stream(stream);
    const int grid = M * C;
#define GAD_CL_FWD(CE_, W_)                                                                          \
    return method == GAD_METHOD_EULER ? cl::launch_fwd_t<CE_, W_, GAD_METHOD_EULER>(a, C, grid, threads, st) \
                                      : cl::launch_fwd_t<CE_, W_, GAD_METHOD_RK4>(a, C, grid, threads, st)
    if (CE == 4 && w == 6) { GAD_CL_FWD(4, 6); }
    if (CE == 4 && w == 7) { GAD_CL_FWD(4, 7); }
    if (CE == 4) { GAD_CL_FWD(4, 3); }
    if (w <= 2) { GAD_CL_FWD(2, 2); }
    GAD_CL_FWD(2, 3);
#undef GAD_CL_FWD
}

namespace gad {
namespace cl {
template <int CE, int W>
int launch_bwd_t(const Args& a, int C, int grid, int threads, cudaStream_t st) {
    auto kern = a.du ? k_cl_bwd<CE, W, true> : k_cl_bwd<CE, W, false>;
    const size_t bytes = make_layout(CE, a.cap_nodes, (threads + 31) / 32).total;
    GAD_CHECK_ARG((int)bytes <= smem_optin_bytes(), "cluster kernel: slab of %d nodes needs %zu B of shared memory",
                  a.cap_nodes, bytes);
    GAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    if (C > 8) GAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    GAD_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    count_launch(1);
    return GAD_OK;
}
}  // namespace cl
}  // namespace gad

/* Deformer backward on cluster-resident meshes (gad_deform_bwd_ell's contract over cluster rows):
 * cotangent g_xphys [N, dim] + saved states [L, N, CE] -> gMu, g_tau (may be NULL), g_x0 (may be NULL), and with the
 * per-mesh bias offset du [M, Lw, CE] of the forward, g_du [M, Lw, CE] (may be NULL).
 * workspace: gad_cluster_workspace_bytes(CE, M, cluster_size, L). */
extern "C" int gad_deform_bwd_cluster(const void* crows_in, const void* crows_out, const int32_t* mesh_ptr, int M,
                                      int max_mesh_nodes, int max_deg, int cluster_size, int64_t N, const float* states,
                                      const float* g_xphys, int dim, int CE, const float* Mu, const float* du, int Lw,
                                      const float* tau, int L, float* gMu, float* g_tau, float* g_x0, float* g_du,
                                      void* workspace, size_t workspace_bytes, void* stream) {
    GAD_CHECK_ARG(crows_in && crows_out && mesh_ptr && states && g_xphys && Mu && tau && gMu && workspace,
                  "gad_deform_bwd_cluster: null pointer");
    GAD_CHECK_ARG(N > 0 && M > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L) && (CE == 2 || CE == 4),
                  "gad_deform_bwd_cluster: N=%lld M=%d L=%d dim=%d CE=%d Lw=%d", (long long)N, M, L, dim, CE, Lw);
    GAD_CHECK_ARG(!g_du || du, "gad_deform_bwd_cluster: g_du needs the bias offset du of the forward");
    const int C = cluster_size;
    GAD_CHECK_ARG(C >= 2 && C <= 16 && (C & (C - 1)) == 0, "gad_deform_bwd_cluster: cluster size %d", C);
    const int grid = M * C;
    GAD_CHECK_ARG(workspace_bytes >= gad_ell_workspace_bytes(CE, grid, L), "gad_deform_bwd_cluster: workspace too small");
    const int S = ((max_mesh_nodes + C - 1) / C + 3) & ~3;
    int threads = ((S + 3) / 4 + 31) / 32 * 32;
    if (threads < 128) threads = 128;
    if (threads > cl::MAXT) threads = cl::MAXT;
    const int NACC = CE * CE + CE + 1, MUSZ = CE * CE + CE;
    float* ws = reinterpret_cast<float*>(workspace);
    ell::Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(crows_in);
    a.ell_out = reinterpret_cast<const uint4*>(crows_out);
    a.tile_ptr = mesh_ptr;
    a.T = grid;
    a.cap_nodes = S;
    a.N = N;
    a.Mu = Mu;
    a.du = du;
    a.tau = tau;
    a.Lw = Lw;
    a.L = L;
    a.dim = dim;
    a.states = const_cast<float*>(states);
    a.g_xphys = g_xphys;
    a.partials = ws;
    a.tau_partials = (g_tau && Lw == 1) ? ws + (size_t)grid * L * NACC : nullptr;
    a.g_x0 = g_x0;
    const int w = cl::slots_for(max_deg);
    cudaStream_t st = as_stream(stream);
    int rc;
    if (CE == 4 && w == 6) rc = cl::launch_bwd_t<4, 6>(a, C, grid, threads, st);
    else if (CE == 4 && w == 7) rc = cl::launch_bwd_t<4, 7>(a, C, grid, threads, st);
    else if (CE == 4) rc = cl::launch_bwd_t<4, 3>(a, C, grid, threads, st);
    else if (w <= 2) rc = cl::launch_bwd_t<2, 2>(a, C, grid, threads, st);
    else rc = cl::launch_bwd_t<2, 3>(a, C, grid, threads, st);
    if (rc) return rc;
    const int slots = Lw > 1 ? L : 1;
    const int ncol = slots * NACC + L + 1;
    cl::k_cl_reduce<<<(ncol + 7) / 8, 256, 0, st>>>(a.partials, grid, slots, NACC, MUSZ, gMu, a.tau_partials, L, g_tau);
    GAD_LAUNCH_CHECK();
    if (g_du) {
        const int n = M * Lw * CE;
        cl::k_cl_du_reduce<<<(n + 127) / 128, 128, 0, st>>>(a.partials, M, C, Lw, slots, NACC, CE, g_du);
        GAD_LAUNCH_CHECK();
    }
    return GAD_OK;
}
