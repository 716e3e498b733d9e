// Streaming kernels: one launch per F-evaluation, one thread per node, state in global memory.
//
// This is the general path of the deformer (any mesh size, any batch shape): it serves meshes too
// large for the mesh-resident kernels of fused_kernels.cu (e.g. the single 200x200 mesh of
// BASELINE config 4), the operator seam `GRAND_plusConv.forward` (src/GRAND_plus.py:204-267) and
// the attention-weight read-out (`stored_alpha`, :253-256).  Per node and F-eval it moves
// 8*CE + 4*deg + 4 bytes (read x_i, write x'_i, col, rowptr; neighbour rows come from L1/L2),
// which is the algorithmic-bytes model of SURVEY 8(d).
#include "common.cuh"
#include "node_math.cuh"

namespace gad {
namespace {

constexpr int TB = 256;

inline unsigned nblocks(int64_t n, int t = TB) { return (unsigned)((n + t - 1) / t); }

// ---- feature assembly + identity encoder (src/GNN.py:225-239, 75-83, 270) -------------------
template <int CE>
__global__ void __launch_bounds__(TB) k_pack(const float* __restrict__ x_comp, const float* __restrict__ f,
                                             const float* __restrict__ uu, const float* __restrict__ f_scale,
                                             const float* __restrict__ uu_scale, int64_t N, int dim,
                                             float* __restrict__ x0) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    Row<CE> r;
#pragma unroll
    for (int c = 0; c < CE; ++c) r.v[c] = 0.f;
    int c = 0;
    for (int d = 0; d < dim && c < CE; ++d, ++c) r.v[c] = x_comp[i * dim + d];
    if (f && c < CE) {
        // the reference divides (f / torch.max(f), GNN.py:232); f_scale holds that max
        r.v[c] = f_scale ? f[i] / f_scale[0] : f[i];
        ++c;
    }
    if (uu && c < CE) {
        r.v[c] = uu_scale ? uu[i] / uu_scale[0] : uu[i];
        ++c;
    }
    store_row<CE>(x0, i, r);
}

// ---- forward stage ------------------------------------------------------------------------
// k = F(y) at every node, then
//     v    = final ? acc_in + k : k
//     out1 = (base ? base : 0) + c1 * v          with c1 = (tau ? tau[0] : 1) * c1_scale
//     out2 = (acc_in ? acc_in : 0) + c2 * k      (RK4 stage accumulator; skipped when null)
//     xphys[i, 0:dim] = out1[0:dim]              (decoder slice, src/GNN.py:298-299; when non-null)
template <int CE>
__global__ void __launch_bounds__(TB) k_stage(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                              int64_t N, const float* __restrict__ y, const float* __restrict__ base,
                                              const float* __restrict__ acc_in, const float* __restrict__ Mu_g,
                                              const float* __restrict__ tau, float c1_scale, float c2, int final_stage,
                                              float* __restrict__ out1, float* __restrict__ out2,
                                              float* __restrict__ xphys, int dim) {
    __shared__ float Mu[CE * CE + CE];
    for (int t = threadIdx.x; t < CE * CE + CE; t += blockDim.x) Mu[t] = Mu_g[t];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const Row<CE> yi = load_row<CE>(y, i);
    const Row<CE> k = node_feval<CE, int32_t>(y, col, rowptr[i], rowptr[i + 1], yi, Mu);
    const float c1 = (tau ? tau[0] : 1.0f) * c1_scale;
    Row<CE> a_in, b_in;
#pragma unroll
    for (int c = 0; c < CE; ++c) a_in.v[c] = b_in.v[c] = 0.f;
    if (acc_in) a_in = load_row<CE>(acc_in, i);
    if (base) b_in = load_row<CE>(base, i);
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

// attention weights of one layer in filtered edge-list order (stored_alpha)
template <int CE>
__global__ void __launch_bounds__(TB) k_alpha(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                              const int32_t* __restrict__ eid, int64_t N, const float* __restrict__ x,
                                              const float* __restrict__ Mu_g, float* __restrict__ alpha) {
    __shared__ float Mu[CE * CE + CE];
    for (int t = threadIdx.x; t < CE * CE + CE; t += blockDim.x) Mu[t] = Mu_g[t];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const Row<CE> xi = load_row<CE>(x, i);
    Row<CE> p;
    SoftmaxStats st;
    const int b = rowptr[i], e_end = rowptr[i + 1];
    node_feval<CE, int32_t>(x, col, b, e_end, xi, Mu, nullptr, &st, &p);
    for (int e = b; e < e_end; ++e) {
        const Row<CE> xj = load_row<CE>(x, (int64_t)col[e]);
        alpha[eid[e]] = gexp(dot<CE>(p, xj) - st.m) * st.rZ;
    }
}

// ---- backward, destination pass -----------------------------------------------------------
// grid-stride over nodes so that the number of weight-gradient partials is bounded.
template <int CE>
__global__ void __launch_bounds__(TB) k_bwd_dst(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                int64_t N, const float* __restrict__ x, const float* __restrict__ gplus,
                                                int gplus_dim,  // < CE: gplus is the [N, dim] cotangent of x_phys
                                                const float* __restrict__ Mu_g, const float* __restrict__ tau,
                                                float a_coef, float b_scale, float* __restrict__ P,
                                                float2* __restrict__ DL, float* __restrict__ gself,
                                                float* __restrict__ partials) {
    constexpr int NACC = CE * CE + CE + 1;
    __shared__ float Mu[CE * CE + CE];
    __shared__ float red[NACC * (TB / 32)];
    for (int t = threadIdx.x; t < CE * CE + CE; t += blockDim.x) Mu[t] = Mu_g[t];
    __syncthreads();
    const float b = (tau ? tau[0] : 1.0f) * b_scale;
    float acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) acc[k] = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const Row<CE> xi = load_row<CE>(x, i);
        Row<CE> gp;
        if (gplus_dim >= CE) {
            gp = load_row<CE>(gplus, i);
        } else {
#pragma unroll
            for (int c = 0; c < CE; ++c) gp.v[c] = (c < gplus_dim) ? gplus[i * gplus_dim + c] : 0.f;
        }
        DstRec<CE> rec;
        const Row<CE> gs = node_bwd_dst<CE, int32_t>(x, col, rowptr[i], rowptr[i + 1], xi, gp, a_coef, b, Mu, &rec,
                                                     acc, &acc[NACC - 1]);
        store_row<CE>(P, i, rec.p);
        DL[i] = make_float2(rec.D, rec.lse);
        store_row<CE>(gself, i, gs);
    }
    block_reduce<NACC>(acc, red, partials + (size_t)blockIdx.x * NACC);
}

// ---- backward, source pass ------------------------------------------------------------------
template <int CE>
__global__ void __launch_bounds__(TB) k_bwd_src(const int32_t* __restrict__ t_rowptr, const int32_t* __restrict__ t_dst,
                                                int64_t N, const float* __restrict__ x, const float* __restrict__ gplus,
                                                int gplus_dim, const float* __restrict__ tau, float b_scale,
                                                const float* __restrict__ P, const float2* __restrict__ DL,
                                                const float* __restrict__ gself, float* __restrict__ gout) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    const float b = (tau ? tau[0] : 1.0f) * b_scale;
    const Row<CE> xj = load_row<CE>(x, j);
    Row<CE> accv;
    if (gplus_dim >= CE) {
        accv = node_bwd_src<CE, int32_t>(P, DL, gplus, t_dst, t_rowptr[j], t_rowptr[j + 1], xj, b);
    } else {
        // first backward layer: the cotangent only has `dim` channels
#pragma unroll
        for (int c = 0; c < CE; ++c) accv.v[c] = 0.f;
        for (int e = t_rowptr[j]; e < t_rowptr[j + 1]; ++e) {
            const int64_t i = t_dst[e];
            const Row<CE> p = load_row<CE>(P, i);
            Row<CE> gp;
#pragma unroll
            for (int c = 0; c < CE; ++c) gp.v[c] = (c < gplus_dim) ? gplus[i * gplus_dim + c] : 0.f;
            const float2 dl = DL[i];
            const float alpha = gexp(dot<CE>(p, xj) - dl.y);
            const float ds = (alpha * LN2_F) * (b * dot<CE>(gp, xj) - dl.x);
            const float ab = alpha * b;
#pragma unroll
            for (int c = 0; c < CE; ++c) accv.v[c] = fmaf(ab, gp.v[c], fmaf(ds, p.v[c], accv.v[c]));
        }
    }
    const Row<CE> gs = load_row<CE>(gself, j);
#pragma unroll
    for (int c = 0; c < CE; ++c) accv.v[c] += gs.v[c];
    store_row<CE>(gout, j, accv);
}

// Fixed-order reduction of per-block partials: out[k] (+)= sum_r partials[r, k].
// One warp per accumulator; lanes stride over rows, then a butterfly -> deterministic.
__global__ void k_reduce_partials(const float* __restrict__ partials, int rows, int nacc, int stride,
                                  float* __restrict__ out, int accumulate) {
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (k >= nacc) return;
    float s = 0.f;
    for (int r = lane; r < rows; r += 32) s += partials[(size_t)r * stride + k];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) out[k] = accumulate ? out[k] + s : s;
}

// ---- mesh loss + cotangent (run_GNN.py:80-84,103-106) ---------------------------------------
// Per-block partial sums of |d| or d^2, d = out[j] - target[i], and the cotangent at out[j].  Without an index map
// j = i.  With one (kOrder, the pde loss) entry i = b * Q + q of `target` pairs with j = b * Q + order[q]: the FEM
// solution stays in evaluation-grid order and the target is in the fine mesh's node order (src/GNN.py:333).
// kCot (gad_mesh_loss kind 2): target[i] is a cotangent c of out[i]; partial sums of out * c, g_out = grad_scale * c.
template <bool kOrder, bool kCot = false>
__device__ __forceinline__ void loss_partials(const float* __restrict__ out, const float* __restrict__ target,
                                              int64_t count, int kind, float grad_scale, float* __restrict__ g_out,
                                              float* __restrict__ partials, const int32_t* __restrict__ order,
                                              int64_t Q) {
    __shared__ float red[TB / 32];
    float acc[1] = {0.f};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t j = i;
        if (kOrder) {
            const int64_t b = i / Q;
            j = b * Q + order[i - b * Q];
        }
        if constexpr (kCot) {
            acc[0] = fmaf(out[j], target[i], acc[0]);
            if (g_out) g_out[j] = grad_scale * target[i];
            continue;
        }
        const float d = out[j] - target[i];
        if (kind == 0) {
            acc[0] += fabsf(d);
            if (g_out) g_out[j] = (d > 0.f ? grad_scale : (d < 0.f ? -grad_scale : 0.f));
        } else {
            acc[0] = fmaf(d, d, acc[0]);
            if (g_out) g_out[j] = 2.f * d * grad_scale;
        }
    }
    block_reduce<1>(acc, red, partials + blockIdx.x);
}

__global__ void __launch_bounds__(TB) k_loss(const float* __restrict__ out, const float* __restrict__ target,
                                             int64_t count, int kind, float grad_scale, float* __restrict__ g_out,
                                             float* __restrict__ partials) {
    loss_partials<false>(out, target, count, kind, grad_scale, g_out, partials, nullptr, 1);
}

__global__ void __launch_bounds__(TB) k_loss_cot(const float* __restrict__ out, const float* __restrict__ cot,
                                                 int64_t count, float grad_scale, float* __restrict__ g_out,
                                                 float* __restrict__ partials) {
    loss_partials<false, true>(out, cot, count, 2, grad_scale, g_out, partials, nullptr, 1);
}

// squared error through the index map (gad_pde_loss)
__global__ void __launch_bounds__(TB) k_loss_ordered(const float* __restrict__ out, const int32_t* __restrict__ order,
                                                     const float* __restrict__ target, int64_t count, int64_t Q,
                                                     float grad_scale, float* __restrict__ g_out,
                                                     float* __restrict__ partials) {
    loss_partials<true>(out, target, count, 1, grad_scale, g_out, partials, order, Q);
}

__global__ void k_loss_final(const float* __restrict__ partials, int rows, float inv_count, float* __restrict__ loss) {
    float s = 0.f;
    for (int r = threadIdx.x; r < rows; r += 32) s += partials[r];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (threadIdx.x == 0) loss[0] = s * inv_count;
}

}  // namespace

// ---- host-side drivers used by api.cu -------------------------------------------------------
int stream_grid_for_partials(int64_t N) {
    const int64_t want = (N + TB - 1) / TB;
    const int64_t cap = (int64_t)sm_count() * 8;
    return (int)(want < cap ? want : cap);
}

template <int CE>
int launch_stage(const int32_t* rowptr, const int32_t* col, int64_t N, const float* y, const float* base,
                 const float* acc_in, const float* Mu, const float* tau, float c1_scale, float c2, int final_stage,
                 float* out1, float* out2, float* xphys, int dim, cudaStream_t st) {
    k_stage<CE><<<nblocks(N), TB, 0, st>>>(rowptr, col, N, y, base, acc_in, Mu, tau, c1_scale, c2, final_stage, out1,
                                           out2, xphys, dim);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

template <int CE>
int stream_forward(const int32_t* rowptr, const int32_t* col, int64_t N, const float* x0, int dim, const float* Mu,
                   int Lw, const float* tau, int L, int method, float* x_phys, float* states, float* ws,
                   cudaStream_t st) {
    const size_t row = (size_t)N * CE;
    const int MUSZ = CE * CE + CE;
    const size_t rowa = align_up(row, 64);
    float* ping[2] = {ws, ws + rowa};
    float* ybuf = ws + 2 * rowa;    // RK4: stage inputs y2 / y4
    float* abuf = ws + 3 * rowa;    // RK4: k1 + 2 k2 + 2 k3
    float* y3buf = ws + 4 * rowa;   // RK4: stage input y3
    const float* cur = x0;
    for (int l = 0; l < L; ++l) {
        const float* Mul = Mu + (size_t)(Lw > 1 ? l : 0) * MUSZ;
        const float* tl = tau + l;
        const bool last = (l == L - 1);
        float* nxt = last ? nullptr : (states ? states + (size_t)(l + 1) * row : ping[l & 1]);
        float* xp = last ? x_phys : nullptr;
        int rc;
        if (method == GAD_METHOD_EULER) {
            rc = launch_stage<CE>(rowptr, col, N, cur, cur, nullptr, Mul, tl, 1.0f, 0.f, 0, nxt, nullptr, xp, dim, st);
            if (rc) return rc;
        } else {
            // k1 = F(x):   y2 = x + h/2 k1,  acc = k1
            rc = launch_stage<CE>(rowptr, col, N, cur, cur, nullptr, Mul, tl, 0.5f, 1.0f, 0, ybuf, abuf, nullptr, dim, st);
            if (rc) return rc;
            // k2 = F(y2):  y3 = x + h/2 k2,  acc += 2 k2
            rc = launch_stage<CE>(rowptr, col, N, ybuf, cur, abuf, Mul, tl, 0.5f, 2.0f, 0, y3buf, abuf, nullptr, dim, st);
            if (rc) return rc;
            // k3 = F(y3):  y4 = x + h k3,    acc += 2 k3
            rc = launch_stage<CE>(rowptr, col, N, y3buf, cur, abuf, Mul, tl, 1.0f, 2.0f, 0, ybuf, abuf, nullptr, dim, st);
            if (rc) return rc;
            // k4 = F(y4):  x' = x + h/6 (acc + k4)
            rc = launch_stage<CE>(rowptr, col, N, ybuf, cur, abuf, Mul, tl, 1.0f / 6.0f, 0.f, 1, nxt, nullptr, xp, dim, st);
            if (rc) return rc;
        }
        cur = nxt;
    }
    return GAD_OK;
}

template <int CE>
int stream_backward(const int32_t* rowptr, const int32_t* col, const int32_t* t_rowptr, const int32_t* t_dst, int64_t N,
                    const float* states, const float* g_xphys, int dim, const float* Mu, int Lw, const float* tau,
                    int L, float a_coef, float* gMu, float* g_tau, float* g_x0, float* ws, cudaStream_t st) {
    constexpr int NACC = CE * CE + CE + 1;
    const int MUSZ = CE * CE + CE;
    const size_t row = (size_t)N * CE;
    const int G = stream_grid_for_partials(N);
    const size_t rowa = align_up(row, 64);
    float* P = ws;
    float* gself = ws + rowa;
    float* gping[2] = {ws + 2 * rowa, ws + 3 * rowa};
    float2* DL = reinterpret_cast<float2*>(ws + 4 * rowa);
    float* partials = ws + 4 * rowa + align_up(2 * (size_t)N, 64);
    GAD_CUDA(cudaMemsetAsync(gMu, 0, (size_t)Lw * MUSZ * sizeof(float), st));
    const float* gcur = g_xphys;
    int gdim = dim < CE ? dim : CE;
    for (int l = L - 1; l >= 0; --l) {
        const float* Mul = Mu + (size_t)(Lw > 1 ? l : 0) * MUSZ;
        const float* xl = states + (size_t)l * row;
        const float* tl = tau ? tau + l : nullptr;
        float* gout = (l == 0 && g_x0) ? g_x0 : gping[l & 1];
        k_bwd_dst<CE><<<G, TB, 0, st>>>(rowptr, col, N, xl, gcur, gdim, Mul, tl, a_coef, 1.0f, P, DL, gself, partials);
        GAD_LAUNCH_CHECK();
        if (l > 0 || g_x0) {
            k_bwd_src<CE><<<nblocks(N), TB, 0, st>>>(t_rowptr, t_dst, N, xl, gcur, gdim, tl, 1.0f, P, DL, gself, gout);
            GAD_LAUNCH_CHECK();
        }
        // G_M, G_u accumulate over layers into the weight set of this layer; g_tau is per layer
        k_reduce_partials<<<(MUSZ + 7) / 8, 256, 0, st>>>(partials, G, MUSZ, NACC, gMu + (size_t)(Lw > 1 ? l : 0) * MUSZ, 1);
        GAD_LAUNCH_CHECK();
        if (g_tau) {
            k_reduce_partials<<<1, 32, 0, st>>>(partials + MUSZ, G, 1, NACC, g_tau + l, 0);
            GAD_LAUNCH_CHECK();
        }
        gcur = gout;
        gdim = CE;
    }
    return GAD_OK;
}

#define GAD_INSTANTIATE(CE)                                                                                          \
    template int stream_forward<CE>(const int32_t*, const int32_t*, int64_t, const float*, int, const float*, int,  \
                                    const float*, int, int, float*, float*, float*, cudaStream_t);                  \
    template int stream_backward<CE>(const int32_t*, const int32_t*, const int32_t*, const int32_t*, int64_t,       \
                                     const float*, const float*, int, const float*, int, const float*, int, float, \
                                     float*, float*, float*, float*, cudaStream_t);
GAD_INSTANTIATE(2)
GAD_INSTANTIATE(4)
GAD_INSTANTIATE(8)

size_t stream_fwd_ws_floats(int64_t N, int CE, int method) {
    // at least 4 rows: the persistent streaming forward keeps two tagged buffers of 2 floats per value there
    return align_up((size_t)N * CE, 64) * (method == GAD_METHOD_RK4 ? 5 : 4) + 64;
}

size_t stream_bwd_ws_floats(int64_t N, int CE) {
    const int NACC = CE * CE + CE + 1;
    // last terms: per-layer step-size partials of the streaming ELL backward (stream_ell.cu: WIDE_TAU_LAYERS = 64), then
    // its per-node t rows of d loss / d du
    const size_t G = (size_t)stream_grid_for_partials(N);
    return align_up((size_t)N * CE, 64) * 5 + align_up(2 * (size_t)N, 64) + align_up(G * NACC, 64) + 64 + G * 64;
}

}  // namespace gad

using namespace gad;

#define GAD_DISPATCH_CE(CE_, FN, ...)                         \
    switch (CE_) {                                            \
        case 2: FN<2> __VA_ARGS__; break;                     \
        case 4: FN<4> __VA_ARGS__; break;                     \
        case 8: FN<8> __VA_ARGS__; break;                     \
        default:                                              \
            gad::set_error("unsupported CE=%d (2, 4, 8)", CE_); \
            return GAD_ERR_UNSUPPORTED;                       \
    }

extern "C" int gad_pack_features(const float* x_comp, const float* f, const float* uu, const float* f_scale,
                                 const float* uu_scale, int64_t N, int dim, int CE, float* x0, void* stream) {
    GAD_CHECK_ARG(x_comp && x0 && N > 0 && dim >= 1 && dim <= 3, "gad_pack_features: bad arguments");
    cudaStream_t st = as_stream(stream);
    GAD_DISPATCH_CE(CE, k_pack, <<<nblocks(N), TB, 0, st>>>(x_comp, f, uu, f_scale, uu_scale, N, dim, x0));
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" int gad_conv_fwd(const int32_t* rowptr, const int32_t* col, const int32_t* eid, int64_t N, int64_t E,
                            const float* x, int CE, const float* Mu, float* res, float* alpha, void* stream) {
    GAD_CHECK_ARG(rowptr && col && x && Mu && N > 0, "gad_conv_fwd: bad arguments");
    GAD_CHECK_ARG(res || alpha, "gad_conv_fwd: nothing to compute");
    GAD_CHECK_ARG(!alpha || eid, "gad_conv_fwd: alpha needs eid");
    cudaStream_t st = as_stream(stream);
    if (res) {
        // res = 0 + 1 * k
        GAD_DISPATCH_CE(CE, k_stage, <<<nblocks(N), TB, 0, st>>>(rowptr, col, N, x, nullptr, nullptr, Mu, nullptr, 1.0f,
                                                                 0.f, 0, res, nullptr, nullptr, 0));
        GAD_LAUNCH_CHECK();
    }
    if (alpha) {
        GAD_DISPATCH_CE(CE, k_alpha, <<<nblocks(N), TB, 0, st>>>(rowptr, col, eid, N, x, Mu, alpha));
        GAD_LAUNCH_CHECK();
    }
    (void)E;
    return GAD_OK;
}

extern "C" int gad_conv_bwd(const int32_t* rowptr, const int32_t* col, const int32_t* t_rowptr, const int32_t* t_dst,
                            int64_t N, int64_t E, const float* x, const float* g_res, int CE, const float* Mu,
                            float* gMu, float* g_x, void* workspace, size_t workspace_bytes, void* stream) {
    GAD_CHECK_ARG(rowptr && col && t_rowptr && t_dst && x && g_res && Mu && gMu && g_x && workspace && N > 0,
                  "gad_conv_bwd: bad arguments");
    GAD_CHECK_ARG(CE == 2 || CE == 4 || CE == 8, "gad_conv_bwd: unsupported CE=%d", CE);
    GAD_CHECK_ARG(workspace_bytes >= stream_bwd_ws_floats(N, CE) * sizeof(float), "gad_conv_bwd: workspace too small");
    cudaStream_t st = as_stream(stream);
    float* ws = reinterpret_cast<float*>(workspace);
    // res = 0*x + 1*(o - x): a = 0, b = 1, one layer, state = x
    int rc = GAD_OK;
    switch (CE) {
        case 2: rc = stream_backward<2>(rowptr, col, t_rowptr, t_dst, N, x, g_res, CE, Mu, 1, nullptr, 1, 0.f, gMu, nullptr, g_x, ws, st); break;
        case 4: rc = stream_backward<4>(rowptr, col, t_rowptr, t_dst, N, x, g_res, CE, Mu, 1, nullptr, 1, 0.f, gMu, nullptr, g_x, ws, st); break;
        case 8: rc = stream_backward<8>(rowptr, col, t_rowptr, t_dst, N, x, g_res, CE, Mu, 1, nullptr, 1, 0.f, gMu, nullptr, g_x, ws, st); break;
    }
    (void)E;
    return rc;
}

extern "C" size_t gad_mesh_loss_workspace_bytes(int64_t count) {
    (void)count;
    return (size_t)(sm_count() * 8 + 8) * sizeof(float);
}

extern "C" int gad_mesh_loss(const float* out, const float* target, int64_t count, int kind, float grad_scale,
                             float* loss, float* g_out, void* workspace, void* stream) {
    GAD_CHECK_ARG(out && target && loss && workspace && count > 0 && kind >= 0 && kind <= 2, "gad_mesh_loss: bad arguments");
    cudaStream_t st = as_stream(stream);
    const int64_t want = (count + TB - 1) / TB;
    const int G = (int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
    float* partials = reinterpret_cast<float*>(workspace);
    if (kind == 2)   // the pseudo-loss <out, c> is a sum, not a mean
        k_loss_cot<<<G, TB, 0, st>>>(out, target, count, grad_scale, g_out, partials);
    else
        k_loss<<<G, TB, 0, st>>>(out, target, count, kind, grad_scale, g_out, partials);
    GAD_LAUNCH_CHECK();
    k_loss_final<<<1, 32, 0, st>>>(partials, G, kind == 2 ? 1.0f : 1.0f / (float)count, loss);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" size_t gad_pde_loss_workspace_bytes(int B, int Q) {
    return gad_mesh_loss_workspace_bytes((int64_t)B * Q);
}

extern "C" int gad_pde_loss(const float* sol, const int32_t* order, const float* target, int B, int Q, float grad_scale,
                            float* loss, float* g_sol, void* workspace, void* stream) {
    GAD_CHECK_ARG(sol && target && loss && workspace, "gad_pde_loss: sol, target, loss and workspace must not be NULL");
    GAD_CHECK_ARG(B > 0 && Q > 0, "gad_pde_loss: B=%d and Q=%d must be positive", B, Q);
    GAD_CHECK_ARG(isfinite(grad_scale), "gad_pde_loss: grad_scale must be finite");
    cudaStream_t st = as_stream(stream);
    const int64_t count = (int64_t)B * Q;
    const int64_t want = (count + TB - 1) / TB;
    const int G = (int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
    float* partials = reinterpret_cast<float*>(workspace);
    // the shared squared-error branch writes 2 * d * s; with s = grad_scale / 2 (exact: a power-of-two scaling) that
    // is d * grad_scale rounded once, i.e. what torch's mse_loss backward writes with grad_scale = 2 / numel
    const float half = 0.5f * grad_scale;
    if (order)
        k_loss_ordered<<<G, TB, 0, st>>>(sol, order, target, count, Q, half, g_sol, partials);
    else
        k_loss<<<G, TB, 0, st>>>(sol, target, count, 1, half, g_sol, partials);
    GAD_LAUNCH_CHECK();
    k_loss_final<<<1, 32, 0, st>>>(partials, G, 1.0f / (float)count, loss);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}
