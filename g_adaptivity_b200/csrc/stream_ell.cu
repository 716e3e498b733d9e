// Streaming ELL kernels: the deformer on meshes too large for one CTA's shared memory (a 60x60 mesh
// already is), one launch per F-evaluation / backward pass, one thread per node, state in global
// memory (L2-resident for the sizes in question).
//
// Same arithmetic as the mesh-resident ELL kernels (ell_math.cuh) -- branch-free rows of W slots,
// all gathers of a row issued back to back, log2-domain softmax with ex2 / lg2 / rcp -- but the
// topology is a "wide" row per node and direction,
//     wide[i] = { int32 j_0 .. j_6, int32 valid }        (32 bytes, two 128-bit loads)
// holding ABSOLUTE neighbour ids (unused slots hold i itself and are masked out), and the
// neighbour rows are gathered from global memory through the read-only path.  Against the CSR
// streaming kernels (stream_kernels.cu: two to three passes over col[] per node, each a dependent
// index load + gather) a node is one pass with no dependent index loads.
//
// The launches of one call form a chain of programmatic dependent launches: every kernel loads what
// does not depend on its predecessor (topology row, folded weights, in the backward destination pass the
// whole softmax recompute from the saved state) BEFORE griddepcontrol.wait, releases its own dependent
// right after the wait (so at most two links are ever resident), and reads whatever the predecessor
// wrote with ld.global.cg -- it was resident while those lines were written, so its L1 may be stale.
// One 200x200 mesh: 2.5 -> 1.8 us per F-evaluation.
//
// Replaces, per layer, `layer(x, edge_index)` + the Euler update (src/GNN.py:273-296) and its
// autograd (src/run_GNN.py:127,130) for graphs of degree <= 7.
#include "common.cuh"
#include "node_math.cuh"

namespace gad {
namespace {

constexpr int TB = 256;
constexpr int WIDE_SLOTS = 7;
constexpr int WIDE_TAU_LAYERS = 64;   // columns of deferred step-size partials the backward workspace holds

inline unsigned nblocks(int64_t n, int t = TB) { return (unsigned)((n + t - 1) / t); }

struct Wide {
    int nb[8];   // nb[7] = validity mask
    __device__ __forceinline__ bool has(int q) const { return (nb[7] >> q) & 1; }
};

__device__ __forceinline__ Wide load_wide(const int4* __restrict__ rows, int64_t i) {
    const int4 a = __ldg(rows + 2 * i), b = __ldg(rows + 2 * i + 1);
    Wide w;
    w.nb[0] = a.x; w.nb[1] = a.y; w.nb[2] = a.z; w.nb[3] = a.w;
    w.nb[4] = b.x; w.nb[5] = b.y; w.nb[6] = b.z; w.nb[7] = b.w;
    return w;
}

template <int CE>
__device__ __forceinline__ Row<CE> ldg_row(const float* __restrict__ base, int64_t i) {
    Row<CE> r;
    if constexpr (CE == 2) {
        const float2 t = __ldg(reinterpret_cast<const float2*>(base) + i);
        r.v[0] = t.x;
        r.v[1] = t.y;
    } else {
        const float4 t = __ldg(reinterpret_cast<const float4*>(base) + i);
        r.v[0] = t.x;
        r.v[1] = t.y;
        r.v[2] = t.z;
        r.v[3] = t.w;
    }
    return r;
}

// State written by the PREVIOUS launch of a programmatic-dependent-launch chain: this kernel is already
// resident while that launch runs, so its L1 cannot be trusted for these buffers -- read through L2.
template <int CE>
__device__ __forceinline__ Row<CE> ldcg_row(const float* base, int64_t i) {
    Row<CE> r;
    if constexpr (CE == 2) {
        const float2 t = __ldcg(reinterpret_cast<const float2*>(base) + i);
        r.v[0] = t.x;
        r.v[1] = t.y;
    } else {
        const float4 t = __ldcg(reinterpret_cast<const float4*>(base) + i);
        r.v[0] = t.x;
        r.v[1] = t.y;
        r.v[2] = t.z;
        r.v[3] = t.w;
    }
    return r;
}

__device__ __forceinline__ void chain_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void chain_release() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Launch of one link of a chain of dependent kernels.  With `dependent` the kernel may become resident
// while its predecessor in the stream still runs (programmatic dependent launch): its prologue -- the
// topology row, the folded weights -- overlaps the predecessor's tail, and it blocks in chain_wait()
// before touching anything the predecessor writes.
inline bool chain_enabled() {
    static const bool on = [] {
        const char* e = getenv("GAD_WIDE_PDL");
        return !(e && e[0] == '0');
    }();
    return on;
}

template <typename... KA, typename... A>
cudaError_t launch_link(void (*kern)(KA...), unsigned G, cudaStream_t st, bool dependent, A... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G);
    cfg.blockDim = dim3(TB);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (dependent && chain_enabled()) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

// cotangent rows: [N, CE], or [N, dim] (dim < CE) for the layer next to the loss
template <int CE>
__device__ __forceinline__ Row<CE> load_gplus(const float* __restrict__ g, int64_t i, int gdim) {
    if (gdim >= CE) return ldg_row<CE>(g, i);
    Row<CE> r;
#pragma unroll
    for (int c = 0; c < CE; ++c) r.v[c] = (c < gdim) ? __ldg(g + i * gdim + c) : 0.f;
    return r;
}

template <int CE>
__device__ __forceinline__ Row<CE> ldcg_gplus(const float* g, int64_t i, int gdim) {
    if (gdim >= CE) return ldcg_row<CE>(g, i);
    Row<CE> r;
#pragma unroll
    for (int c = 0; c < CE; ++c) r.v[c] = (c < gdim) ? __ldcg(g + i * gdim + c) : 0.f;
    return r;
}

// ---- wide rows from the (row-sorted) CSR / CSC walk arrays ---------------------------------------
__global__ void __launch_bounds__(TB) k_build_wide(const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                                                   int64_t N, int4* __restrict__ rows, int32_t* __restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int b = ptr[i], deg = ptr[i + 1] - b;
    int v[8];
#pragma unroll
    for (int q = 0; q < WIDE_SLOTS; ++q) v[q] = (q < deg) ? idx[b + q] : (int)i;
    v[7] = (deg >= WIDE_SLOTS) ? 0x7f : ((1 << deg) - 1);
    if (deg > WIDE_SLOTS) {
        atomicAdd(bad, 1);
        v[7] = 0;
    }
    rows[2 * i] = make_int4(v[0], v[1], v[2], v[3]);
    rows[2 * i + 1] = make_int4(v[4], v[5], v[6], v[7]);
}

// ---- forward stage (same contract as k_stage of stream_kernels.cu) -------------------------------
//     k = F(y);  v = final ? acc_in + k : k;  out1 = base + c1 v;  out2 = acc_in + c2 k
// du (or null): the bias offset of this weight set for mesh 0, du + m * du_stride for mesh m = i / nm.
template <int CE, int W>
__global__ void __launch_bounds__(TB) k_wide_stage(const int4* __restrict__ rows, int64_t N, const float* __restrict__ y,
                                                   const float* __restrict__ base, const float* __restrict__ acc_in,
                                                   const float* __restrict__ Mu_g, const float* __restrict__ du,
                                                   int du_stride, int64_t nm, const float* __restrict__ tau,
                                                   float c1_scale, float c2, int final_stage, float* __restrict__ out1,
                                                   float* __restrict__ out2, float* __restrict__ xphys, int dim) {
    __shared__ float Mu[CE * CE + CE];
    for (int t = threadIdx.x; t < CE * CE + CE; t += blockDim.x) Mu[t] = Mu_g[t];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const Wide w = load_wide(rows, i);
    const float tau0 = tau ? __ldg(tau) : 1.0f;
    const float* dui = du ? du + (i / nm) * du_stride : nullptr;
    // everything above is independent of the previous launch; everything below reads what it wrote
    chain_wait();
    chain_release();
    const Row<CE> yi = ldcg_row<CE>(y, i);
    // ---- F(y) at node i: project, gather, softmax, aggregate (ell_math.cuh: ell_feval) ----
    const Row<CE> p = project_du<CE>(Mu, dui, yi);
    Row<CE> xj[W];
    float s[W];
    float m = -3.0e38f;
#pragma unroll
    for (int q = 0; q < W; ++q) {
        xj[q] = ldcg_row<CE>(y, (int64_t)w.nb[q]);
        const float d = dot<CE>(p, xj[q]);
        s[q] = w.has(q) ? d : -CUDART_INF_F;
        m = fmaxf(m, s[q]);
    }
    float Z = 0.f;
    Row<CE> o = zero_row<CE>();
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const float e = ex2_approx(s[q] - m);
        Z += e;
#pragma unroll
        for (int c = 0; c < CE; ++c) o.v[c] = fmaf(e, xj[q].v[c], o.v[c]);
    }
    const float rZ = (w.nb[7] != 0) ? rcp_refined(Z) : 0.f;
    Row<CE> k;
#pragma unroll
    for (int c = 0; c < CE; ++c) k.v[c] = fmaf(o.v[c], rZ, -yi.v[c]);
    // ---- stage combination ----
    const float c1 = tau0 * c1_scale;
    Row<CE> a_in = zero_row<CE>(), b_in = zero_row<CE>();
    if (acc_in) a_in = ldcg_row<CE>(acc_in, i);
    if (base) b_in = (base == y) ? yi : ldcg_row<CE>(base, i);
    Row<CE> o1;
#pragma unroll
    for (int c = 0; c < CE; ++c) {
        const float v = final_stage ? a_in.v[c] + k.v[c] : k.v[c];
        o1.v[c] = fmaf(c1, v, b_in.v[c]);
    }
    if (out1) store_row<CE>(out1, i, o1);
    if (out2) {
        Row<CE> o2;
#pragma unroll
        for (int c = 0; c < CE; ++c) o2.v[c] = fmaf(c2, k.v[c], a_in.v[c]);
        store_row<CE>(out2, i, o2);
    }
    if (xphys) {
        for (int d = 0; d < dim && d < CE; ++d) xphys[i * dim + d] = o1.v[d];
    }
}

// ---- persistent forward: all L steps (x 4 RK4 stages) of one call in ONE launch --------------------------------
// For graphs whose nodes fit the co-resident threads of the GPU (one 200x200 mesh: 157 CTAs on 148 SMs) the chain of
// one launch per F-evaluation above spends half of every link on the launch hand-over, and a grid barrier per
// F-evaluation (release fence + counter + acquire poll) was measured at the same 2 us.  Here neither exists:
//   * every thread keeps its node -- topology row, state x, RK4 accumulator -- in registers for the whole call;
//   * a CTA owns S = 256 consecutive nodes and keeps the stage input y of its WINDOW (the strips of the CTAs within
//     r = ceil(reach / S) of it, reach = max |j - i| over the edges) in shared memory: all gathers are LDS;
//   * after each F-evaluation a thread publishes its new row to one of two global (L2-resident) buffers as
//     (value, epoch) pairs, each pair one 64-bit element of a 256-bit relaxed vector access (the idea of NCCL's LL
//     protocol: a datum is valid when the tag that travels in the same atomic word matches -- no fence, no barrier),
//     and the CTA polls the 2 r S halo rows of its window into shared memory.
// A CTA waits only for the CTAs within r of it, so the machine synchronises locally.  Two buffers suffice because the
// windows are symmetric: B overwrites its epoch-e rows with epoch e+2 only after it has read the epoch-(e+1) rows of
// every CTA within r, each of which published them after it finished reading B's epoch-e rows.
// The arithmetic is k_wide_stage's, expression for expression: results are bit-identical to the chain.  The launch
// is cooperative (all CTAs co-resident or the launch fails); a poll that sees no progress for 2 s traps.
// A row travels as CE (value, epoch) pairs, each ONE 64-bit element of a vector access: whatever the hardware does
// with the vector as a whole, a 64-bit element is a single-copy-atomic access, so a value can never be seen with
// another epoch's tag.
__device__ __forceinline__ unsigned long long tagged(float v, unsigned tag) {
    return ((unsigned long long)tag << 32) | (unsigned long long)__float_as_uint(v);
}

template <int CE>
__device__ __forceinline__ void publish_row(float* buf, int64_t i, const Row<CE>& r, unsigned tag) {
    if constexpr (CE == 4) {      // one 32-byte store (256-bit accesses exist from sm_100 on)
        asm volatile("st.relaxed.gpu.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(buf + i * 8), "l"(tagged(r.v[0], tag)),
                     "l"(tagged(r.v[1], tag)), "l"(tagged(r.v[2], tag)), "l"(tagged(r.v[3], tag))
                     : "memory");
    } else {
        asm volatile("st.relaxed.gpu.global.v2.b64 [%0], {%1, %2};" ::"l"(buf + i * 4), "l"(tagged(r.v[0], tag)),
                     "l"(tagged(r.v[1], tag))
                     : "memory");
    }
}

// One poll of a row: true when every (value, epoch) pair carries `tag`.
template <int CE>
__device__ __forceinline__ bool try_row(const float* p, unsigned tag, Row<CE>& r) {
    unsigned long long v[CE];
    if constexpr (CE == 4) {
        asm volatile("ld.relaxed.gpu.global.v4.b64 {%0, %1, %2, %3}, [%4];"
                     : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3])
                     : "l"(p)
                     : "memory");
    } else {
        asm volatile("ld.relaxed.gpu.global.v2.b64 {%0, %1}, [%2];" : "=l"(v[0]), "=l"(v[1]) : "l"(p) : "memory");
    }
    bool ok = true;
#pragma unroll
    for (int c = 0; c < CE; ++c) {
        r.v[c] = __uint_as_float((unsigned)v[c]);
        ok = ok && (unsigned)(v[c] >> 32) == tag;
    }
    return ok;
}

template <int CE>
__device__ __forceinline__ Row<CE> lds_row(const float* sm, int j) {
    Row<CE> r;
    if constexpr (CE == 2) {
        const float2 t = reinterpret_cast<const float2*>(sm)[j];
        r.v[0] = t.x;
        r.v[1] = t.y;
    } else {
        const float4 t = reinterpret_cast<const float4*>(sm)[j];
        r.v[0] = t.x;
        r.v[1] = t.y;
        r.v[2] = t.z;
        r.v[3] = t.w;
    }
    return r;
}

template <int CE>
__device__ __forceinline__ void sts_row(float* sm, int j, const Row<CE>& r) {
    if constexpr (CE == 2) reinterpret_cast<float2*>(sm)[j] = make_float2(r.v[0], r.v[1]);
    else reinterpret_cast<float4*>(sm)[j] = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
}

// F(y) at one node, neighbours at LOCAL window indices (same expression order as k_wide_stage)
template <int CE, int W>
__device__ __forceinline__ Row<CE> window_feval(const float* Mu, const float* dui, const int* nbl, int valid,
                                                const float* ysm, const Row<CE>& yi) {
    const Row<CE> p = project_du<CE>(Mu, dui, yi);
    Row<CE> xj[W];
    float s[W];
    float m = -3.0e38f;
#pragma unroll
    for (int q = 0; q < W; ++q) {
        xj[q] = lds_row<CE>(ysm, nbl[q]);
        const float d = dot<CE>(p, xj[q]);
        s[q] = ((valid >> q) & 1) ? d : -CUDART_INF_F;
        m = fmaxf(m, s[q]);
    }
    float Z = 0.f;
    Row<CE> o = zero_row<CE>();
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const float e = ex2_approx(s[q] - m);
        Z += e;
#pragma unroll
        for (int c = 0; c < CE; ++c) o.v[c] = fmaf(e, xj[q].v[c], o.v[c]);
    }
    const float rZ = (valid != 0) ? rcp_refined(Z) : 0.f;
    Row<CE> k;
#pragma unroll
    for (int c = 0; c < CE; ++c) k.v[c] = fmaf(o.v[c], rZ, -yi.v[c]);
    return k;
}

#ifndef GAD_PERSIST_MINB
#define GAD_PERSIST_MINB 3      // co-resident CTAs per SM the register budget allows (capacity = 148 x this x 256 nodes)
#endif
template <int CE, int W>
__global__ void __launch_bounds__(TB, GAD_PERSIST_MINB) k_wide_persist(const int4* __restrict__ rows, int64_t N, int r,
                                                     const float* __restrict__ x0, const float* __restrict__ Mu_g,
                                                     const float* __restrict__ du, int64_t nm, int Lw,
                                                     const float* __restrict__ tau, int L, int method, float* tbuf0,
                                                     float* tbuf1, float* states, float* __restrict__ xphys, int dim) {
    constexpr int MUSZ = CE * CE + CE;
    constexpr int S = TB;
    __shared__ float Mu[MUSZ];
    extern __shared__ float4 ysm4[];
    float* ysm = reinterpret_cast<float*>(ysm4);             // [(2 r + 1) S][CE], row w <-> node wlo + w
    const int64_t n0 = (int64_t)blockIdx.x * S;
    const int64_t wlo = n0 - (int64_t)r * S;
    const int64_t i = n0 + threadIdx.x;
    const bool live = i < N;
    const int64_t ic = live ? i : n0;                        // idle threads of the last CTA shadow its first node
    const int own = r * S + threadIdx.x;                     // this thread's row of the window
    const int halo = 2 * r * S;
    int nbl[W], valid;
    {
        const Wide w = load_wide(rows, ic);
#pragma unroll
        for (int q = 0; q < W; ++q) nbl[q] = (int)((int64_t)w.nb[q] - wlo);
        valid = live ? w.nb[7] : 0;
    }
    Row<CE> x = ldg_row<CE>(x0, ic);
    // Needed part of the halo (window rows), widened so that every strip of the window contributes at least one row:
    // that keeps the dependencies between CTAs symmetric, which is what makes two buffers enough (see above).
    __shared__ int need[2];
    if (threadIdx.x == 0) {
        need[0] = r * S - 1 - (r - 1) * S;                   // last row of the farthest strip on the left  (= S - 1)
        need[1] = (r + 1) * S + (r - 1) * S;                 // first row of the farthest strip on the right (= 2 r S)
    }
    __syncthreads();
    if (live) {
        int lo = own, hi = own;
#pragma unroll
        for (int q = 0; q < W; ++q) {
            lo = min(lo, nbl[q]);
            hi = max(hi, nbl[q]);
        }
        atomicMin(&need[0], lo);
        atomicMax(&need[1], hi);
    }
    __syncthreads();
    const int need_lo = max(need[0], 0), need_hi = min(need[1], halo + S - 1);
    const int n_left = r * S - need_lo, n_need = n_left + (need_hi - (r + 1) * S + 1);
    // window of the initial state (an input of the call: plain loads)
    for (int h = threadIdx.x; h < halo + S; h += TB) {
        const int64_t j = wlo + h;
        if (j >= 0 && j < N) sts_row<CE>(ysm, h, ldg_row<CE>(x0, j));
    }
    unsigned epoch = 0;
    const size_t row = (size_t)N * CE;
    // This thread's share of the needed halo rows (two per pass; one pass when the halo has at most 2 TB rows): window
    // row and offset into a tagged buffer, fixed for the whole call.
    int hrow[2];
    int64_t hoff[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int k = threadIdx.x + u * TB;
        const int wr = k < n_left ? need_lo + k : (r + 1) * S + (k - n_left);
        const int64_t j = wlo + wr;
        hrow[u] = (k < n_need && j >= 0 && j < N) ? wr : -1;
        hoff[u] = j * (2 * CE);
    }
    const bool one_pass = n_need <= 2 * TB;
    auto poll_pair = [&](const float* buf, const int* wr, const int64_t* off) {
        bool pending[2] = {wr[0] >= 0, wr[1] >= 0};
        unsigned long long t0 = 0;
        for (unsigned spins = 1; pending[0] || pending[1]; ++spins) {
            Row<CE> t[2];
            bool ok[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) ok[u] = pending[u] && try_row<CE>(buf + off[u], epoch, t[u]);
#pragma unroll
            for (int u = 0; u < 2; ++u)
                if (ok[u]) {
                    sts_row<CE>(ysm, wr[u], t[u]);
                    pending[u] = false;
                }
            if ((spins & 0xfff) == 0) {                      // a neighbour that never publishes must not hang the device
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (t0 == 0) t0 = now;
                else if (now - t0 > 2000000000ull) __trap();
            }
        }
    };
    // hand the next stage input to the window: own row to shared memory and to the world, halo rows from the world
    auto exchange = [&](const Row<CE>& y) {
        ++epoch;
        float* buf = (epoch & 1) ? tbuf1 : tbuf0;
        if (live) publish_row<CE>(buf, i, y, epoch);
        __syncthreads();                                     // every thread has finished reading the old window
        sts_row<CE>(ysm, own, y);
        if (one_pass) {
            poll_pair(buf, hrow, hoff);
        } else {
            for (int h = threadIdx.x; h < n_need; h += 2 * TB) {
                int wr[2];
                int64_t off[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int k = h + u * TB;
                    wr[u] = k < n_left ? need_lo + k : (r + 1) * S + (k - n_left);
                    const int64_t j = wlo + wr[u];
                    if (!(k < n_need && j >= 0 && j < N)) wr[u] = -1;
                    off[u] = j * (2 * CE);
                }
                poll_pair(buf, wr, off);
            }
        }
        __syncthreads();
    };
    // One flat loop over the F-evaluations (ONE copy of the F-evaluation and of the exchange in the instruction
    // stream: with two warps per scheduler nothing hides instruction fetches).  RK4 stage sg of step l:
    //   sg < 3: y = x + c1 k, acc += c2 k          sg = 3: x += (tau / 6) (acc + k), y = x
    const bool rk4 = method == GAD_METHOD_RK4;
    const int per_step = rk4 ? 4 : 1, E = L * per_step;
    Row<CE> y = x, acc = zero_row<CE>();
    float tau0 = 0.f;
    const float* dui = nullptr;                              // bias offset of this node's mesh and the current weight set
#pragma unroll 1
    for (int e = 0; e < E; ++e) {
        const int l = rk4 ? (e >> 2) : e, sg = rk4 ? (e & 3) : 3;
        if (sg == 0 || !rk4) {
            if (e == 0 || Lw > 1) {
                __syncthreads();
                for (int t = threadIdx.x; t < MUSZ; t += blockDim.x) Mu[t] = Mu_g[(size_t)(Lw > 1 ? l : 0) * MUSZ + t];
                __syncthreads();
                if (du) dui = du + ((ic / nm) * Lw + (Lw > 1 ? l : 0)) * CE;
            }
            tau0 = __ldg(tau + l);
        }
        const Row<CE> k = window_feval<CE, W>(Mu, dui, nbl, valid, ysm, y);
        if (sg < 3) {
            const float c1 = tau0 * (sg == 2 ? 1.0f : 0.5f), c2 = (sg == 0 ? 1.0f : 2.0f);
#pragma unroll
            for (int c = 0; c < CE; ++c) {
                y.v[c] = fmaf(c1, k.v[c], x.v[c]);
                acc.v[c] = fmaf(c2, k.v[c], acc.v[c]);
            }
        } else {
            const float c1 = tau0 * (rk4 ? 1.0f / 6.0f : 1.0f);
#pragma unroll
            for (int c = 0; c < CE; ++c) {
                x.v[c] = fmaf(c1, rk4 ? acc.v[c] + k.v[c] : k.v[c], x.v[c]);
                y.v[c] = x.v[c];
                acc.v[c] = 0.f;
            }
            if (e == E - 1) {
                if (live)
                    for (int d = 0; d < dim && d < CE; ++d) xphys[i * dim + d] = x.v[d];
            } else if (states && live) {
                store_row<CE>(states + (size_t)(l + 1) * row, i, x);
            }
        }
        if (e < E - 1) exchange(y);
    }
}

// ---- backward, destination pass (contract of k_bwd_dst; math of ell_bwd_dst) ----------------------
// grid-stride over nodes so that the number of weight-gradient partials is bounded.
template <int CE, int W>
__global__ void __launch_bounds__(TB) k_wide_bwd_dst(const int4* __restrict__ rows, int64_t N, const float* __restrict__ x,
                                                     const float* __restrict__ gplus, int gplus_dim,
                                                     const float* __restrict__ Mu_g, const float* __restrict__ du,
                                                     int du_stride, int64_t nm, const float* __restrict__ tau,
                                                     float a_coef, float* __restrict__ P, float2* __restrict__ DL,
                                                     float* __restrict__ gself, float* __restrict__ partials,
                                                     int accumulate, float* __restrict__ tau_part, int tau_stride,
                                                     float* __restrict__ trows) {
    constexpr int NACC = CE * CE + CE + 1;
    __shared__ float Mu[CE * CE + CE];
    __shared__ float red[NACC * (TB / 32)];
    __shared__ float blk[NACC];
    for (int t = threadIdx.x; t < CE * CE + CE; t += blockDim.x) Mu[t] = Mu_g[t];
    __syncthreads();
    const float b = tau ? tau[0] : 1.0f;
    float acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) acc[k] = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const Wide w = load_wide(rows, i);
        const Row<CE> xi = ldg_row<CE>(x, i);
        const bool any = w.nb[7] != 0;
        const Row<CE> p = project_du<CE>(Mu, du ? du + (i / nm) * du_stride : nullptr, xi);
        Row<CE> xj[W];
        float s[W];
        float m = -3.0e38f;
#pragma unroll
        for (int q = 0; q < W; ++q) {
            xj[q] = ldg_row<CE>(x, (int64_t)w.nb[q]);
            const float d = dot<CE>(p, xj[q]);
            s[q] = w.has(q) ? d : -CUDART_INF_F;
            m = fmaxf(m, s[q]);
        }
        float Z = 0.f;
        Row<CE> o = zero_row<CE>();
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
        // the recompute above reads only the saved states; the cotangent comes from the previous launch
        chain_wait();
        chain_release();
        const Row<CE> gp = ldcg_gplus<CE>(gplus, i, gplus_dim);
        Row<CE> go;
#pragma unroll
        for (int c = 0; c < CE; ++c) go.v[c] = b * gp.v[c];
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
        float gb = 0.f;
#pragma unroll
        for (int c = 0; c < CE; ++c) gb = fmaf(gp.v[c], o.v[c] - xi.v[c], gb);
        acc[NACC - 1] += gb;
#pragma unroll
        for (int aa = 0; aa < CE; ++aa)
#pragma unroll
            for (int bb = 0; bb < CE; ++bb) acc[aa * CE + bb] = fmaf(xi.v[aa], t.v[bb], acc[aa * CE + bb]);
#pragma unroll
        for (int bb = 0; bb < CE; ++bb) acc[CE * CE + bb] += t.v[bb];
        if (trows) {   // t_i of every pass of the weight set, summed per node: d loss / d du of its mesh (k_wide_du_reduce)
            Row<CE> tt = t;
            if (accumulate) {
                const Row<CE> prev = ldcg_row<CE>(trows, i);
#pragma unroll
                for (int c = 0; c < CE; ++c) tt.v[c] = prev.v[c] + t.v[c];
            }
            store_row<CE>(trows, i, tt);
        }
        const Row<CE> Mt = apply_M<CE>(Mu, t);
        Row<CE> gs;
#pragma unroll
        for (int c = 0; c < CE; ++c) gs.v[c] = fmaf(a_coef - b, gp.v[c], Mt.v[c]);
        store_row<CE>(P, i, p);
        DL[i] = make_float2(D, lse);
        store_row<CE>(gself, i, gs);
    }
    // per-block partial row: (G_M, G_u) accumulate over the layers of a shared weight set (same block,
    // same order every time: deterministic), the step-size column is per layer
    chain_wait();
    block_reduce<NACC>(acc, red, blk);
    if (threadIdx.x < NACC) {
        float* dst = partials + (size_t)blockIdx.x * NACC + threadIdx.x;
        *dst = (accumulate && threadIdx.x < NACC - 1) ? __ldcg(dst) + blk[threadIdx.x] : blk[threadIdx.x];
        // step-size partials of ALL layers side by side ([block][layer]) when the reduction is deferred
        if (tau_part && threadIdx.x == NACC - 1) tau_part[(size_t)blockIdx.x * tau_stride] = blk[NACC - 1];
    }
}

// ---- backward, source pass (contract of k_bwd_src; math of ell_bwd_src) -----------------------------
template <int CE, int W>
__global__ void __launch_bounds__(TB) k_wide_bwd_src(const int4* __restrict__ rows_out, int64_t N,
                                                     const float* __restrict__ x, const float* __restrict__ gplus,
                                                     int gplus_dim, const float* __restrict__ tau,
                                                     const float* __restrict__ P, const float2* __restrict__ DL,
                                                     const float* __restrict__ gself, float* __restrict__ gout) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    const float b = tau ? tau[0] : 1.0f;
    const Wide w = load_wide(rows_out, j);
    const Row<CE> xj = ldg_row<CE>(x, j);
    // the out-edge row and the saved state do not depend on the destination pass; its outputs do
    chain_wait();
    chain_release();
    Row<CE> p[W], gp[W];
    float2 dl[W];
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const int64_t i = (int64_t)w.nb[q];
        p[q] = ldcg_row<CE>(P, i);
        gp[q] = ldcg_gplus<CE>(gplus, i, gplus_dim);
        dl[q] = __ldcg(DL + i);
    }
    Row<CE> accv = ldcg_row<CE>(gself, j);
#pragma unroll
    for (int q = 0; q < W; ++q) {
        const float sv = dot<CE>(p[q], xj) - dl[q].y;
        const float alpha = ex2_approx(w.has(q) ? sv : -CUDART_INF_F);
        const float ds = (alpha * LN2_F) * (b * dot<CE>(gp[q], xj) - dl[q].x);
        const float ab = alpha * b;
#pragma unroll
        for (int c = 0; c < CE; ++c) accv.v[c] = fmaf(ab, gp[q].v[c], fmaf(ds, p[q].v[c], accv.v[c]));
    }
    store_row<CE>(gout, j, accv);
}

// ---- RK4 backward on the streaming kernels: bookkeeping between the four vjp passes of a step ------------------
//   a_out = ca_g * g + ca_gy * gy   (cotangent of the next stage to differentiate, in units of 1 / tau)
//   gs    = (first ? g : gs) + gy    (running cotangent of the step input)
// g is [N, gdim] (gdim < CE next to the loss), everything else [N, CE].
template <int CE>
__global__ void __launch_bounds__(TB) k_wide_rk4_comb(int64_t N, const float* __restrict__ g, int gdim,
                                                      const float* __restrict__ gy, float ca_g, float ca_gy,
                                                      float* __restrict__ a_out, float* __restrict__ gs, int first) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const Row<CE> gi = load_gplus<CE>(g, i, gdim);
    Row<CE> yi = zero_row<CE>();
    if (gy) yi = load_row<CE>(gy, i);
    if (a_out) {
        Row<CE> a;
#pragma unroll
        for (int c = 0; c < CE; ++c) a.v[c] = fmaf(ca_gy, yi.v[c], ca_g * gi.v[c]);
        store_row<CE>(a_out, i, a);
    }
    if (gs) {
        Row<CE> o = first ? gi : load_row<CE>(gs, i);
#pragma unroll
        for (int c = 0; c < CE; ++c) o.v[c] += yi.v[c];
        store_row<CE>(gs, i, o);
    }
}

// Fixed-order reduction of the per-block partials (one warp per accumulator): out[k] (+)= sum_r part[r, k].
__global__ void k_wide_reduce(const float* __restrict__ partials, int rows, int nacc, int stride, float* __restrict__ out,
                              int accumulate) {
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (k >= nacc) return;
    double s = 0.0;
    for (int r = lane; r < rows; r += 32) s += (double)partials[(size_t)r * stride + k];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) out[k] = accumulate ? out[k] + (float)s : (float)s;
}

// d loss / d du[b, lw] = sum of the t rows of mesh b (nodes b nm .. (b + 1) nm - 1): one CTA per mesh, lane-strided fp64
// sums and a fixed-order tree over the block -- the same bits every run.
template <int CE>
__global__ void __launch_bounds__(TB) k_wide_du_reduce(const float* __restrict__ trows, int64_t nm, int Lw, int lw,
                                                       float* __restrict__ g_du) {
    __shared__ double red[TB][CE];
    const int b = blockIdx.x, tid = threadIdx.x;
    double s[CE];
#pragma unroll
    for (int c = 0; c < CE; ++c) s[c] = 0.0;
    for (int64_t i = tid; i < nm; i += TB) {
        const Row<CE> t = load_row<CE>(trows, (int64_t)b * nm + i);
#pragma unroll
        for (int c = 0; c < CE; ++c) s[c] += (double)t.v[c];
    }
#pragma unroll
    for (int c = 0; c < CE; ++c) red[tid][c] = s[c];
    __syncthreads();
    for (int w = TB / 2; w > 0; w >>= 1) {
        if (tid < w)
#pragma unroll
            for (int c = 0; c < CE; ++c) red[tid][c] += red[tid + w][c];
        __syncthreads();
    }
    if (tid < CE) g_du[((size_t)b * Lw + lw) * CE + tid] = (float)red[0][tid];
}

int grid_for_partials(int64_t N) {
    const int64_t want = (N + TB - 1) / TB;
    const int64_t cap = (int64_t)sm_count() * 8;
    return (int)(want < cap ? want : cap);
}

// Can the persistent kernel take this call?  G CTAs of TB nodes with a window of (2 r + 1) TB rows in shared memory
// must all be co-resident on the current device (cooperative launch).  GAD_WIDE_PERSIST=0 keeps the chain of
// dependent launches (read per call: the tests switch between the two routes).
constexpr size_t PERSIST_SMEM_MAX = 96 * 1024;

template <int CE, int W>
bool persist_fits(unsigned G, int r, size_t smem) {
    const char* e = getenv("GAD_WIDE_PERSIST");
    if ((e && e[0] == '0') || r < 0 || smem > PERSIST_SMEM_MAX) return false;
    auto kern = k_wide_persist<CE, W>;
    static thread_local int cached_dev = -1, sms = 0, coop = 0;
    static thread_local size_t cached_smem = 0;
    static thread_local int per_sm = 0;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    if (dev != cached_dev || smem != cached_smem) {
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) != cudaSuccess ||
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PERSIST_SMEM_MAX) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TB, smem) != cudaSuccess)
            return false;
        cached_dev = dev;
        cached_smem = smem;
    }
    const bool fits = coop && (int)G <= sms * per_sm;
    if (getenv("GAD_TRACE_ROUTE"))
        fprintf(stderr, "[gad] k_wide_persist<%d,%d>: G=%u r=%d smem=%zu capacity=%d CTAs -> %s\n", CE, W, G, r, smem,
                sms * per_sm, fits ? "one launch" : "launch chain");
    return fits;
}

template <int CE, int W>
int persist_capacity_t(int64_t reach, int64_t* nodes) {
    const int r = (int)((reach + TB - 1) / TB);
    const size_t smem = (size_t)(2 * r + 1) * TB * CE * sizeof(float);
    int64_t lo = 0, hi = 1 << 20;                    // largest G that fits, by bisection over the cached occupancy
    if (!persist_fits<CE, W>(1, r, smem)) {
        *nodes = 0;
        return GAD_OK;
    }
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) / 2;
        (persist_fits<CE, W>((unsigned)mid, r, smem) ? lo : hi) = mid;
    }
    *nodes = lo * TB;
    return GAD_OK;
}

int slots_for(int max_deg) { return max_deg <= 2 ? 2 : (max_deg <= 3 ? 3 : (max_deg <= 6 ? 6 : 7)); }

template <int CE, int W>
int wide_forward_t(const int4* rows, int64_t N, int64_t reach, const float* x0, int dim, const float* Mu, const float* du,
                   int64_t nm, int Lw, const float* tau, int L, int method, float* x_phys, float* states, float* ws,
                   cudaStream_t st) {
    const size_t row = (size_t)N * CE;
    const int MUSZ = CE * CE + CE;
    const size_t rowa = align_up(row, 64);
    float* ping[2] = {ws, ws + rowa};
    float* ybuf = ws + 2 * rowa;    // RK4: stage inputs y2 / y4
    float* abuf = ws + 3 * rowa;    // RK4: k1 + 2 k2 + 2 k3
    float* y3buf = ws + 4 * rowa;   // RK4: stage input y3
    const float* cur = x0;
    const unsigned G = nblocks(N);
    const int r = reach < 0 ? -1 : (int)((reach + TB - 1) / TB);
    const size_t smem = (size_t)(2 * (r < 0 ? 0 : r) + 1) * TB * CE * sizeof(float);
    if ((L > 1 || method == GAD_METHOD_RK4) && persist_fits<CE, W>(G, r, smem)) {
        // ONE cooperative launch for the whole call.  The two tagged buffers (2 floats per state value) live in the
        // workspace and start with tag 0 everywhere; epochs count from 1.
        float* tb0 = ws;
        float* tb1 = ws + 2 * rowa;
        GAD_CUDA(cudaMemsetAsync(ws, 0, 4 * rowa * sizeof(float), st));
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(G);
        cfg.blockDim = dim3(TB);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        GAD_CUDA(cudaLaunchKernelEx(&cfg, k_wide_persist<CE, W>, rows, N, r, x0, Mu, du, nm, Lw, tau, L, method, tb0, tb1,
                                    states, x_phys, dim));
        count_launch(1);
        return GAD_OK;
    }
    const int dus = Lw * CE;
    for (int l = 0; l < L; ++l) {
        const float* Mul = Mu + (size_t)(Lw > 1 ? l : 0) * MUSZ;
        const float* dul = du ? du + (size_t)(Lw > 1 ? l : 0) * CE : nullptr;
        const float* tl = tau + l;
        const bool last = (l == L - 1);
        float* nxt = last ? nullptr : (states ? states + (size_t)(l + 1) * row : ping[l & 1]);
        float* xp = last ? x_phys : nullptr;
        if (method == GAD_METHOD_EULER) {
            GAD_CUDA(launch_link(k_wide_stage<CE, W>, G, st, l > 0, rows, N, cur, cur, (const float*)nullptr, Mul, dul, dus, nm,
                                 tl, 1.0f, 0.f, 0, nxt, (float*)nullptr, xp, dim));
            count_launch(1);
        } else {
            // classical RK4 on F(y) = A(y) y - y (stream_kernels.cu: stream_forward)
            GAD_CUDA(launch_link(k_wide_stage<CE, W>, G, st, l > 0, rows, N, cur, cur, (const float*)nullptr, Mul, dul, dus, nm,
                                 tl, 0.5f, 1.0f, 0, ybuf, abuf, (float*)nullptr, dim));
            GAD_CUDA(launch_link(k_wide_stage<CE, W>, G, st, true, rows, N, (const float*)ybuf, cur, (const float*)abuf,
                                 Mul, dul, dus, nm, tl, 0.5f, 2.0f, 0, y3buf, abuf, (float*)nullptr, dim));
            GAD_CUDA(launch_link(k_wide_stage<CE, W>, G, st, true, rows, N, (const float*)y3buf, cur, (const float*)abuf,
                                 Mul, dul, dus, nm, tl, 1.0f, 2.0f, 0, ybuf, abuf, (float*)nullptr, dim));
            GAD_CUDA(launch_link(k_wide_stage<CE, W>, G, st, true, rows, N, (const float*)ybuf, cur, (const float*)abuf,
                                 Mul, dul, dus, nm, tl, 1.0f / 6.0f, 0.f, 1, nxt, (float*)nullptr, xp, dim));
            count_launch(4);
        }
        cur = nxt;
    }
    return GAD_OK;
}

template <int CE, int W>
int wide_backward_t(const int4* rows_in, const int4* rows_out, int64_t N, const float* states, const float* g_xphys,
                    int dim, const float* Mu, const float* du, int M, int Lw, const float* tau, int L, float* gMu,
                    float* g_tau, float* g_x0, float* g_du, float* ws, cudaStream_t st) {
    constexpr int NACC = CE * CE + CE + 1;
    const int MUSZ = CE * CE + CE;
    const size_t row = (size_t)N * CE;
    const int G = grid_for_partials(N);
    const size_t rowa = align_up(row, 64);
    float* P = ws;
    float* gself = ws + rowa;
    float* gping[2] = {ws + 2 * rowa, ws + 3 * rowa};
    float2* DL = reinterpret_cast<float2*>(ws + 4 * rowa);
    float* partials = ws + 4 * rowa + align_up(2 * (size_t)N, 64);
    GAD_CUDA(cudaMemsetAsync(gMu, 0, (size_t)Lw * MUSZ * sizeof(float), st));
    const float* gcur = g_xphys;
    int gdim = dim;
    // Step-size partials of all layers are kept side by side and reduced once at the end, so that (with one
    // shared weight set) nothing is launched between the passes and the whole backward is one chain of
    // dependent launches; the workspace holds WIDE_TAU_LAYERS columns.
    const bool defer_tau = g_tau && L <= WIDE_TAU_LAYERS;
    float* taup = partials + align_up((size_t)G * NACC, 64);
    // per-node t rows of the passes of one weight set (d loss / d du, reduced per mesh): after the step-size columns
    float* trows = g_du ? taup + (size_t)G * WIDE_TAU_LAYERS : nullptr;
    const int64_t nm = N / M;
    const int dus = Lw * CE;
    bool first = true;
    for (int l = L - 1; l >= 0; --l) {
        const float* Mul = Mu + (size_t)(Lw > 1 ? l : 0) * MUSZ;
        const float* dul = du ? du + (size_t)(Lw > 1 ? l : 0) * CE : nullptr;
        const float* xl = states + (size_t)l * row;
        const float* tl = tau + l;
        float* gout = (l == 0 && g_x0) ? g_x0 : gping[l & 1];
        const bool shared_w = (Lw == 1);
        GAD_CUDA(launch_link(k_wide_bwd_dst<CE, W>, (unsigned)G, st, !first, rows_in, N, xl, gcur, gdim, Mul, dul, dus, nm,
                             tl, 1.0f, P, DL, gself, partials, (shared_w && l < L - 1) ? 1 : 0,
                             defer_tau ? taup + l : (float*)nullptr, L, trows));
        count_launch(1);
        first = false;
        if (l > 0 || g_x0) {
            GAD_CUDA(launch_link(k_wide_bwd_src<CE, W>, nblocks(N), st, true, rows_out, N, xl, gcur, gdim, tl,
                                 (const float*)P, (const float2*)DL, (const float*)gself, gout));
            count_launch(1);
        }
        if (!shared_w || l == 0) {   // shared weights: one reduction of the accumulated partials at the end
            k_wide_reduce<<<(MUSZ + 7) / 8, 256, 0, st>>>(partials, G, MUSZ, NACC, gMu + (size_t)(shared_w ? 0 : l) * MUSZ, 1);
            GAD_LAUNCH_CHECK();
            if (trows) {
                k_wide_du_reduce<CE><<<M, TB, 0, st>>>(trows, nm, Lw, shared_w ? 0 : l, g_du);
                GAD_LAUNCH_CHECK();
            }
        }
        if (g_tau && !defer_tau) {
            k_wide_reduce<<<1, 32, 0, st>>>(partials + MUSZ, G, 1, NACC, g_tau + l, 0);
            GAD_LAUNCH_CHECK();
        }
        gcur = gout;
        gdim = CE;
    }
    if (defer_tau) {
        k_wide_reduce<<<(L + 7) / 8, 256, 0, st>>>(taup, G, L, L, g_tau, 0);
        GAD_LAUNCH_CHECK();
    }
    return GAD_OK;
}

}  // namespace

size_t stream_fwd_ws_floats(int64_t N, int CE, int method);
size_t stream_bwd_ws_floats(int64_t N, int CE);

}  // namespace gad

using namespace gad;

size_t wide_bwd_rk4_ws_floats(int64_t N, int CE) {
    const int NACC = CE * CE + CE + 1;
    // nine state rows, DL, the per-block partials, the per-node t rows of d loss / d du
    return align_up((size_t)N * CE, 64) * 10 + align_up(2 * (size_t)N, 64) +
           align_up((size_t)grid_for_partials(N) * NACC, 64) + 64;
}

// Backward through L classical RK4 steps of F(y) = A(y) y - y on the streaming kernels, from the saved step inputs
// x^0 .. x^{L-1}.  Per step, in reverse: recompute the stage inputs y2, y3, y4 (three k_wide_stage launches), then four
// vjp passes (k_wide_bwd_dst + k_wide_bwd_src with a_coef = 0: gout = tau J(y_s)^T a) on the cotangents
//   a4 = g / 6,  a3 = g / 3 + gy4,  a2 = g / 3 + gy3 / 2,  a1 = g / 6 + gy2 / 2      (a_s = dL/dk_s / tau)
// and g(step input) = g + gy1 + gy2 + gy3 + gy4.  The weight-gradient partials accumulate over the four passes (and,
// with one shared weight set, over all steps) in the same blocks in the same order: deterministic.  No step-size
// gradient (learn_step is an Euler feature, as in k_ell_bwd_rk4).
template <int CE, int W>
int wide_backward_rk4_t(const int4* rows_in, const int4* rows_out, int64_t N, const float* states, const float* g_xphys,
                        int dim, const float* Mu, const float* du, int M, int Lw, const float* tau, int L, float* gMu,
                        float* g_x0, float* g_du, float* ws, cudaStream_t st) {
    constexpr int NACC = CE * CE + CE + 1;
    const int MUSZ = CE * CE + CE;
    const size_t row = (size_t)N * CE;
    const int G = grid_for_partials(N);
    const unsigned GN = nblocks(N);
    const size_t rowa = align_up(row, 64);
    float* P = ws;
    float* gself = ws + rowa;
    float* a = ws + 2 * rowa;
    float* gy = ws + 3 * rowa;
    float* gsb[2] = {ws + 4 * rowa, ws + 5 * rowa};
    float* yb[3] = {ws + 6 * rowa, ws + 7 * rowa, ws + 8 * rowa};       // y2, y3, y4
    float2* DL = reinterpret_cast<float2*>(ws + 9 * rowa);
    float* partials = ws + 9 * rowa + align_up(2 * (size_t)N, 64);
    float* trows = g_du ? partials + align_up((size_t)G * NACC, 64) : nullptr;
    const int64_t nm = N / M;
    const int dus = Lw * CE;
    GAD_CUDA(cudaMemsetAsync(gMu, 0, (size_t)Lw * MUSZ * sizeof(float), st));
    const float* gcur = g_xphys;
    int gdim = dim;
    const bool shared_w = (Lw == 1);
    bool first_of_set = true;
    static const float ca_g[4] = {1.0f / 6.0f, 1.0f / 3.0f, 1.0f / 3.0f, 1.0f / 6.0f};      // of a1 .. a4
    for (int l = L - 1; l >= 0; --l) {
        const float* Mul = Mu + (size_t)(Lw > 1 ? l : 0) * MUSZ;
        const float* dul = du ? du + (size_t)(Lw > 1 ? l : 0) * CE : nullptr;
        const float* xl = states + (size_t)l * row;
        const float* tl = tau + l;
        float* gs = (l == 0 && g_x0) ? g_x0 : gsb[l & 1];
        // stage inputs: y2 = x + tau/2 F(x), y3 = x + tau/2 F(y2), y4 = x + tau F(y3)
        const float* yin = xl;
        for (int sgi = 0; sgi < 3; ++sgi) {
            GAD_CUDA(launch_link(k_wide_stage<CE, W>, GN, st, false, rows_in, N, yin, xl, (const float*)nullptr, Mul, dul, dus,
                                 nm, tl, sgi == 2 ? 1.0f : 0.5f, 0.f, 0, yb[sgi], (float*)nullptr, (float*)nullptr, dim));
            yin = yb[sgi];
        }
        count_launch(3);
        if (!shared_w) first_of_set = true;
        k_wide_rk4_comb<CE><<<GN, TB, 0, st>>>(N, gcur, gdim, (const float*)nullptr, ca_g[3], 0.f, a, (float*)nullptr, 0);
        GAD_LAUNCH_CHECK();
        for (int sgi = 3; sgi >= 0; --sgi) {
            const float* ys = sgi == 0 ? xl : yb[sgi - 1];
            GAD_CUDA(launch_link(k_wide_bwd_dst<CE, W>, (unsigned)G, st, false, rows_in, N, ys, (const float*)a, CE, Mul, dul,
                                 dus, nm, tl, 0.0f, P, DL, gself, partials, first_of_set ? 0 : 1, (float*)nullptr, 0, trows));
            first_of_set = false;
            GAD_CUDA(launch_link(k_wide_bwd_src<CE, W>, GN, st, false, rows_out, N, ys, (const float*)a, CE, tl,
                                 (const float*)P, (const float2*)DL, (const float*)gself, gy));
            count_launch(2);
            // next cotangent (a3 = g/3 + gy4, a2 = g/3 + gy3/2, a1 = g/6 + gy2/2) and the running sum g + sum gy
            k_wide_rk4_comb<CE><<<GN, TB, 0, st>>>(N, gcur, gdim, (const float*)gy, sgi > 0 ? ca_g[sgi - 1] : 0.f,
                                                 sgi == 3 ? 1.0f : 0.5f, sgi > 0 ? a : (float*)nullptr, gs, sgi == 3);
            GAD_LAUNCH_CHECK();
        }
        if (!shared_w || l == 0) {
            k_wide_reduce<<<(MUSZ + 7) / 8, 256, 0, st>>>(partials, G, MUSZ, NACC, gMu + (size_t)(shared_w ? 0 : l) * MUSZ, 1);
            GAD_LAUNCH_CHECK();
            if (trows) {
                k_wide_du_reduce<CE><<<M, TB, 0, st>>>(trows, nm, Lw, shared_w ? 0 : l, g_du);
                GAD_LAUNCH_CHECK();
            }
        }
        gcur = gs;
        gdim = CE;
    }
    return GAD_OK;
}

#define GAD_WIDE_DISPATCH(FN, ...)                                                     \
    do {                                                                               \
        const int w__ = slots_for(max_deg);                                            \
        if (CE == 2 && w__ == 2) return FN<2, 2>(__VA_ARGS__);                         \
        if (CE == 2 && w__ == 3) return FN<2, 3>(__VA_ARGS__);                         \
        if (CE == 2 && w__ == 6) return FN<2, 6>(__VA_ARGS__);                         \
        if (CE == 2 && w__ == 7) return FN<2, 7>(__VA_ARGS__);                         \
        if (CE == 4 && w__ == 2) return FN<4, 2>(__VA_ARGS__);                         \
        if (CE == 4 && w__ == 3) return FN<4, 3>(__VA_ARGS__);                         \
        if (CE == 4 && w__ == 6) return FN<4, 6>(__VA_ARGS__);                         \
        if (CE == 4 && w__ == 7) return FN<4, 7>(__VA_ARGS__);                         \
        set_error("wide kernels: no instantiation for CE=%d max_deg=%d", CE, max_deg); \
        return GAD_ERR_UNSUPPORTED;                                                    \
    } while (0)

extern "C" int gad_graph_build_wide(const int32_t* ptr, const int32_t* idx, int64_t N, void* wide_rows, int32_t* info,
                                    void* stream) {
    GAD_CHECK_ARG(ptr && idx && wide_rows && info && N > 0, "gad_graph_build_wide: bad arguments");
    k_build_wide<<<nblocks(N), TB, 0, as_stream(stream)>>>(ptr, idx, N, reinterpret_cast<int4*>(wide_rows),
                                                          info + GAD_INFO_ELL_BAD);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

// The per-mesh bias offset du [M, Lw, CE] (NULL: none) of the streaming entry points: M meshes of N / M nodes each,
// node i in mesh i / (N / M).
#define GAD_WIDE_CHECK_DU(FN)                                                                                      \
    GAD_CHECK_ARG(!du || (M > 0 && N % M == 0), FN ": du needs M > 0 meshes of equal size (N=%lld, M=%d)", (long long)N, M)

extern "C" int gad_deform_fwd_wide(const void* wide_in, int64_t N, int max_deg, int64_t reach, const float* x0, int dim, int CE,
                                   const float* Mu, const float* du, int M, int Lw, const float* tau, int L, int method,
                                   float* x_phys, float* states, void* workspace, size_t workspace_bytes, void* stream) {
    GAD_CHECK_ARG(wide_in && x0 && Mu && tau && x_phys && workspace, "gad_deform_fwd_wide: null pointer");
    GAD_CHECK_ARG(N > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L) && max_deg >= 0 && max_deg <= WIDE_SLOTS,
                  "gad_deform_fwd_wide: N=%lld L=%d dim=%d CE=%d Lw=%d max_deg=%d", (long long)N, L, dim, CE, Lw, max_deg);
    GAD_CHECK_ARG(method == GAD_METHOD_EULER || method == GAD_METHOD_RK4, "gad_deform_fwd_wide: unknown method %d", method);
    GAD_CHECK_ARG(!states || states == x0, "gad_deform_fwd_wide: when states is given, x0 must alias states[0]");
    GAD_CHECK_ARG(workspace_bytes >= stream_fwd_ws_floats(N, CE, method) * sizeof(float),
                  "gad_deform_fwd_wide: workspace too small");
    GAD_WIDE_CHECK_DU("gad_deform_fwd_wide");
    const int4* rows = reinterpret_cast<const int4*>(wide_in);
    float* ws = reinterpret_cast<float*>(workspace);
    cudaStream_t st = as_stream(stream);
    const int64_t nm = du ? N / M : N;
    GAD_WIDE_DISPATCH(wide_forward_t, rows, N, reach, x0, dim, Mu, du, nm, Lw, tau, L, method, x_phys, states, ws, st);
}

extern "C" size_t gad_deform_bwd_wide_rk4_workspace_bytes(int64_t N, int CE) {
    return wide_bwd_rk4_ws_floats(N, CE) * sizeof(float);
}

extern "C" int gad_deform_bwd_wide_rk4(const void* wide_in, const void* wide_out, int64_t N, int max_deg,
                                       const float* states, const float* g_xphys, int dim, int CE, const float* Mu,
                                       const float* du, int M, int Lw, const float* tau, int L, float* gMu, float* g_x0,
                                       float* g_du, void* workspace, size_t workspace_bytes, void* stream) {
    GAD_CHECK_ARG(wide_in && wide_out && states && g_xphys && Mu && tau && gMu && workspace,
                  "gad_deform_bwd_wide_rk4: null pointer");
    GAD_CHECK_ARG(N > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L) && max_deg >= 0 && max_deg <= WIDE_SLOTS,
                  "gad_deform_bwd_wide_rk4: N=%lld L=%d dim=%d CE=%d Lw=%d max_deg=%d", (long long)N, L, dim, CE, Lw, max_deg);
    GAD_CHECK_ARG(workspace_bytes >= wide_bwd_rk4_ws_floats(N, CE) * sizeof(float),
                  "gad_deform_bwd_wide_rk4: workspace too small");
    GAD_WIDE_CHECK_DU("gad_deform_bwd_wide_rk4");
    GAD_CHECK_ARG(!g_du || du, "gad_deform_bwd_wide_rk4: g_du needs the bias offset du of the forward");
    const int4* rin = reinterpret_cast<const int4*>(wide_in);
    const int4* rout = reinterpret_cast<const int4*>(wide_out);
    float* ws = reinterpret_cast<float*>(workspace);
    cudaStream_t st = as_stream(stream);
    GAD_WIDE_DISPATCH(wide_backward_rk4_t, rin, rout, N, states, g_xphys, dim, Mu, du, du ? M : 1, Lw, tau, L, gMu, g_x0, g_du,
                      ws, st);
}

extern "C" int64_t gad_wide_persist_nodes(int CE, int max_deg, int64_t reach) {
    int64_t nodes = 0;
    if (reach < 0 || max_deg < 0 || max_deg > WIDE_SLOTS || (CE != 2 && CE != 4)) return 0;
    auto run = [&]() -> int { GAD_WIDE_DISPATCH(persist_capacity_t, reach, &nodes); };
    return run() == GAD_OK ? nodes : 0;
}

extern "C" int gad_deform_bwd_wide(const void* wide_in, const void* wide_out, int64_t N, int max_deg,
                                   const float* states, const float* g_xphys, int dim, int CE, const float* Mu,
                                   const float* du, int M, int Lw, const float* tau, int L, float* gMu, float* g_tau,
                                   float* g_x0, float* g_du, void* workspace, size_t workspace_bytes, void* stream) {
    GAD_CHECK_ARG(wide_in && wide_out && states && g_xphys && Mu && tau && gMu && workspace,
                  "gad_deform_bwd_wide: null pointer");
    GAD_CHECK_ARG(N > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L) && max_deg >= 0 && max_deg <= WIDE_SLOTS,
                  "gad_deform_bwd_wide: N=%lld L=%d dim=%d CE=%d Lw=%d max_deg=%d", (long long)N, L, dim, CE, Lw, max_deg);
    GAD_CHECK_ARG(workspace_bytes >= stream_bwd_ws_floats(N, CE) * sizeof(float), "gad_deform_bwd_wide: workspace too small");
    GAD_WIDE_CHECK_DU("gad_deform_bwd_wide");
    GAD_CHECK_ARG(!g_du || du, "gad_deform_bwd_wide: g_du needs the bias offset du of the forward");
    const int4* rin = reinterpret_cast<const int4*>(wide_in);
    const int4* rout = reinterpret_cast<const int4*>(wide_out);
    float* ws = reinterpret_cast<float*>(workspace);
    cudaStream_t st = as_stream(stream);
    GAD_WIDE_DISPATCH(wide_backward_t, rin, rout, N, states, g_xphys, dim, Mu, du, du ? M : 1, Lw, tau, L, gMu, g_tau, g_x0,
                      g_du, ws, st);
}
