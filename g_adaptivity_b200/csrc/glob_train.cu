// Global CNN features in the training step: the per-mesh offset of the folded bias and its adjoint.
//
// The CNN output g_b of mesh b (GNN._global_bias_offsets, src/GNN.py:242-268) reaches the deformer kernels as
//     du_b[lw, z] = c * sum_g (Wq[lw]^T Wk[lw])[z0 + g, z] * g_b[g]        (z < live, zero up to CE)
// with c = fold_scale(inv_temp, C), z0 = the node-varying input channels, g < n_g = the global channels the identity
// encoder keeps.  The backward reads G_b = dL/ddu_b from the per-tile partials of the deformer's backward (one mesh
// per tile) and returns
//     dL/dg_b[g]          = c * sum_lw sum_z Mg[lw, g, z] G_b[lw, z]                         (for gad_cnn_bwd)
//     dL/dWq[lw][k, z0+g] += c * sum_z Wk[lw][k, z] H[lw, g, z]
//     dL/dWk[lw][k, z]    += c * sum_g Wq[lw][k, z0+g] H[lw, g, z],   H[lw, g, z] = sum_b g_b[g] G_b[lw, z]
// H is summed over the meshes in fp64 in mesh order: no atomics, bit-reproducible.
#include "common.cuh"
#include "tail_math.cuh"

namespace gad {
namespace {

constexpr int GB_THREADS = 128;
constexpr int GB_MAX_G = 32;      // n_g <= 2 * Co <= 2 * 16 (glob_cnn.cu: CNN_MAX_C)
constexpr int GB_MAX_CE = 8;
constexpr int GB_MAX_LW = 16;

struct GlobArgs {
    const float* g_f;     // [B, Co] or null
    const float* g_uu;    // [B, Co] or null
    const float* Wq;      // [Lw, C, C]
    const float* Wk;      // [Lw, C, C]
    int B, Co, n_g, Lw, C, z0, live, CE;
    float c;
};

// channel g of cat[g_f | g_uu] of mesh b
__device__ __forceinline__ float glob_feat(const GlobArgs& a, int b, int g) {
    if (a.g_f) {
        if (g < a.Co) return a.g_f[(size_t)b * a.Co + g];
        g -= a.Co;
    }
    return a.g_uu[(size_t)b * a.Co + g];
}

// Mg[lw][g][z] = c * (Wq[lw]^T Wk[lw])[z0 + g, z] into shared memory (all threads; ends with a barrier)
__device__ void glob_mg(const GlobArgs& a, float* Mg) {
    const int n = a.Lw * a.n_g * a.live;
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
        const int z = t % a.live, g = (t / a.live) % a.n_g, lw = t / (a.live * a.n_g);
        const float* wq = a.Wq + (size_t)lw * a.C * a.C + a.z0 + g;
        const float* wk = a.Wk + (size_t)lw * a.C * a.C + z;
        float s = 0.f;
        for (int k = 0; k < a.C; ++k) s = fmaf(wq[(size_t)k * a.C], wk[(size_t)k * a.C], s);
        Mg[t] = a.c * s;
    }
    __syncthreads();
}

// one CTA per mesh: du [B, Lw, CE]
__global__ void __launch_bounds__(GB_THREADS) k_glob_bias_fwd(const GlobArgs a, float* __restrict__ du) {
    __shared__ float Mg[GB_MAX_LW * GB_MAX_G * GB_MAX_CE];
    __shared__ float g[GB_MAX_G];
    const int b = blockIdx.x;
    for (int t = threadIdx.x; t < a.n_g; t += blockDim.x) g[t] = glob_feat(a, b, t);
    glob_mg(a, Mg);
    for (int t = threadIdx.x; t < a.Lw * a.CE; t += blockDim.x) {
        const int z = t % a.CE, lw = t / a.CE;
        float s = 0.f;
        if (z < a.live)
            for (int k = 0; k < a.n_g; ++k) s = fmaf(Mg[(lw * a.n_g + k) * a.live + z], g[k], s);
        du[(size_t)b * a.Lw * a.CE + t] = s;
    }
}

// G_b[lw, z]: entries CE*CE + z of the partial row (b, lw) -- [T, slots, CE*CE + CE + 1], slots = Lw (include/gadapt.h)
__device__ __forceinline__ float glob_gdu(const GlobArgs& a, const float* part, int b, int lw, int z) {
    const int nacc = a.CE * a.CE + a.CE + 1;
    return part[((size_t)b * a.Lw + lw) * nacc + a.CE * a.CE + z];
}

// one CTA per mesh: dL/dg_b into g_out_f / g_out_uu [B, Co] (zero for the truncated outputs)
__global__ void __launch_bounds__(GB_THREADS) k_glob_bias_bwd_g(const GlobArgs a, const float* __restrict__ part,
                                                               float* __restrict__ g_out_f, float* __restrict__ g_out_uu) {
    __shared__ float Mg[GB_MAX_LW * GB_MAX_G * GB_MAX_CE];
    const int b = blockIdx.x;
    glob_mg(a, Mg);
    const int n_out = (a.g_f ? a.Co : 0) + (a.g_uu ? a.Co : 0);
    for (int gi = threadIdx.x; gi < n_out; gi += blockDim.x) {
        float s = 0.f;
        if (gi < a.n_g)
            for (int lw = 0; lw < a.Lw; ++lw)
                for (int z = 0; z < a.live; ++z) s = fmaf(Mg[(lw * a.n_g + gi) * a.live + z], glob_gdu(a, part, b, lw, z), s);
        float* out = (a.g_f && gi < a.Co) ? g_out_f + (size_t)b * a.Co + gi
                                          : g_out_uu + (size_t)b * a.Co + (a.g_f ? gi - a.Co : gi);
        *out = s;
    }
}

// one CTA per weight set: H = sum_b g_b G_b^T (fp64, mesh order), then the du terms of gWq / gWk
__global__ void __launch_bounds__(GB_THREADS) k_glob_bias_bwd_w(const GlobArgs a, const float* __restrict__ part,
                                                               float* __restrict__ gWq, float* __restrict__ gWk) {
    __shared__ double H[GB_MAX_G * GB_MAX_CE];
    const int lw = blockIdx.x;
    for (int t = threadIdx.x; t < a.n_g * a.live; t += blockDim.x) {
        const int z = t % a.live, g = t / a.live;
        double s = 0.0;
        for (int b = 0; b < a.B; ++b) s += (double)glob_feat(a, b, g) * (double)glob_gdu(a, part, b, lw, z);
        H[t] = s;
    }
    __syncthreads();
    const size_t off = (size_t)lw * a.C * a.C;
    const float* wq = a.Wq + off;
    const float* wk = a.Wk + off;
    for (int t = threadIdx.x; t < a.C * a.n_g; t += blockDim.x) {
        const int g = t % a.n_g, k = t / a.n_g;
        double s = 0.0;
        for (int z = 0; z < a.live; ++z) s += (double)wk[(size_t)k * a.C + z] * H[g * a.live + z];
        gWq[off + (size_t)k * a.C + a.z0 + g] += (float)(a.c * s);
    }
    for (int t = threadIdx.x; t < a.C * a.live; t += blockDim.x) {
        const int z = t % a.live, k = t / a.live;
        double s = 0.0;
        for (int g = 0; g < a.n_g; ++g) s += (double)wq[(size_t)k * a.C + a.z0 + g] * H[g * a.live + z];
        gWk[off + (size_t)k * a.C + z] += (float)(a.c * s);
    }
}

// max |u| over n values: the bits of non-negative floats order like the values, so an integer max is exact and
// independent of the order in which blocks arrive
__global__ void k_absmax(const float* __restrict__ u, int64_t n, unsigned int* __restrict__ out) {
    float m = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        m = fmaxf(m, fabsf(u[i]));
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, d));
    if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));
}

// NaN-propagating max, as torch.max: a NaN on either side wins
__device__ __forceinline__ float nan_max(float a, float b) { return (a > b || a != a) ? a : b; }

// signed max over n values (gnn_normalize: f / torch.max(f)).  `out` starts as 0xffffffff, a bit pattern below every
// candidate in both orders used here: a non-negative float (sign bit clear) wins an integer max against any negative
// one, and among negative floats the smaller unsigned bits are the larger value.  NaN enters as the positive quiet
// NaN, which is above +inf as an integer.  The result does not depend on the order in which warps arrive.
__global__ void k_batch_max(const float* __restrict__ x, int64_t n, unsigned int* __restrict__ out) {
    float m = -INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        m = nan_max(m, x[i]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) m = nan_max(m, __shfl_xor_sync(0xffffffffu, m, d));
    if ((threadIdx.x & 31) == 0) {
        const unsigned int bits = (m != m) ? 0x7fc00000u : __float_as_uint(m);
        if (bits & 0x80000000u) atomicMin(out, bits);
        else atomicMax(reinterpret_cast<int*>(out), (int)bits);
    }
}

// learnable temperature: the logits of weight set l are divided by temp[l], i.e. its folded weights are scaled by
// 1 / temp[l], rounded as functional.DeformFunction.forward does (an fp32 reciprocal, then a multiply)
__global__ void k_temp_fold(const float* __restrict__ Mu, const float* __restrict__ temp, int Lw, int S,
                            float* __restrict__ Mu_eff) {
    for (int t = threadIdx.x; t < Lw * S; t += blockDim.x) {
        const float inv = 1.0f / temp[t / S];
        Mu_eff[t] = Mu[t] * inv;
    }
}

// one CTA per weight set: g_temp[l] = -sum_j gMu[l, j] * Mu_eff[l, j] / temp[l] (fixed-order tree, no atomics) and
// gMu_base[l] = gMu[l] / temp[l] (DeformFunction.backward)
constexpr int TF_THREADS = 128;
__global__ void __launch_bounds__(TF_THREADS) k_temp_fold_bwd(const float* __restrict__ gMu, const float* __restrict__ Mu_eff,
                                                              const float* __restrict__ temp, int S,
                                                              float* __restrict__ gMu_base, float* __restrict__ g_temp) {
    __shared__ float red[TF_THREADS];
    const int l = blockIdx.x;
    const float t = temp[l];
    const float* g = gMu + (size_t)l * S;
    const float* mu = Mu_eff + (size_t)l * S;
    float s = 0.f;
    for (int j = threadIdx.x; j < S; j += TF_THREADS) {
        s = fmaf(g[j], mu[j], s);
        gMu_base[(size_t)l * S + j] = g[j] / t;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = TF_THREADS / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) g_temp[l] = -red[0] / t;
}

int glob_fill(GlobArgs& a, const char* who, const float* g_f, const float* g_uu, int B, int Co, int n_g,
              const float* Wq, const float* Wk, int Lw, int C, int z0, int live, int CE, float inv_temp) {
    GAD_CHECK_ARG((g_f || g_uu) && Wq && Wk, "%s: null pointer", who);
    const int n_src = (g_f ? 1 : 0) + (g_uu ? 1 : 0);
    GAD_CHECK_ARG(B > 0 && Co > 0 && Lw > 0 && Lw <= GB_MAX_LW && C > 0, "%s: B=%d Co=%d Lw=%d C=%d", who, B, Co, Lw, C);
    GAD_CHECK_ARG(n_g >= 1 && n_g <= n_src * Co && n_g <= GB_MAX_G,
                  "%s: n_g=%d global channels from %d outputs of %d channels (at most %d)", who, n_g, n_src, Co, GB_MAX_G);
    GAD_CHECK_ARG(CE >= 1 && CE <= GB_MAX_CE && live >= 1 && live <= CE, "%s: live=%d CE=%d", who, live, CE);
    GAD_CHECK_ARG(z0 >= 0 && z0 + n_g <= C && live <= C, "%s: z0=%d + n_g=%d exceeds C=%d (live=%d)", who, z0, n_g, C, live);
    a.g_f = g_f, a.g_uu = g_uu, a.Wq = Wq, a.Wk = Wk;
    a.B = B, a.Co = Co, a.n_g = n_g, a.Lw = Lw, a.C = C, a.z0 = z0, a.live = live, a.CE = CE;
    a.c = (float)tail::fold_scale(inv_temp, C);
    return GAD_OK;
}

}  // namespace
}  // namespace gad

using namespace gad;

extern "C" int gad_glob_bias_fwd(const float* g_f, const float* g_uu, int B, int Co, int n_g, const float* Wq,
                                 const float* Wk, int Lw, int C, int z0, int live, int CE, float inv_temp, float* du,
                                 void* stream) {
    GlobArgs a{};
    int rc = glob_fill(a, "gad_glob_bias_fwd", g_f, g_uu, B, Co, n_g, Wq, Wk, Lw, C, z0, live, CE, inv_temp);
    if (rc) return rc;
    GAD_CHECK_ARG(du, "gad_glob_bias_fwd: null output");
    k_glob_bias_fwd<<<B, GB_THREADS, 0, as_stream(stream)>>>(a, du);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" int gad_glob_bias_bwd(const float* g_f, const float* g_uu, int B, int Co, int n_g, const float* Wq,
                                 const float* Wk, int Lw, int C, int z0, int live, int CE, float inv_temp,
                                 const void* workspace, size_t workspace_bytes, float* g_out_f, float* g_out_uu,
                                 float* gWq, float* gWk, void* stream) {
    GlobArgs a{};
    int rc = glob_fill(a, "gad_glob_bias_bwd", g_f, g_uu, B, Co, n_g, Wq, Wk, Lw, C, z0, live, CE, inv_temp);
    if (rc) return rc;
    GAD_CHECK_ARG(workspace && gWq && gWk && (!g_f || g_out_f) && (!g_uu || g_out_uu), "gad_glob_bias_bwd: null pointer");
    const size_t need = (size_t)B * Lw * (CE * CE + CE + 1) * sizeof(float);
    GAD_CHECK_ARG(workspace_bytes >= need, "gad_glob_bias_bwd: the workspace holds %zu B, the per-tile partials of %d "
                                           "meshes need %zu B", workspace_bytes, B, need);
    const float* part = reinterpret_cast<const float*>(workspace);
    cudaStream_t st = as_stream(stream);
    k_glob_bias_bwd_g<<<B, GB_THREADS, 0, st>>>(a, part, g_out_f, g_out_uu);
    GAD_LAUNCH_CHECK();
    k_glob_bias_bwd_w<<<Lw, GB_THREADS, 0, st>>>(a, part, gWq, gWk);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" int gad_absmax(const float* u, int64_t n, float* out, void* stream) {
    GAD_CHECK_ARG(u && out && n > 0, "gad_absmax: null pointer or empty input");
    cudaStream_t st = as_stream(stream);
    GAD_CUDA(cudaMemsetAsync(out, 0, sizeof(float), st));
    const int64_t blocks = (n + 256 * 8 - 1) / (256 * 8);
    const int grid = (int)(blocks < 4LL * sm_count() ? blocks : 4LL * sm_count());
    k_absmax<<<grid, 256, 0, st>>>(u, n, reinterpret_cast<unsigned int*>(out));
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" int gad_batch_max(const float* x, int64_t n, float* out, void* stream) {
    GAD_CHECK_ARG(x && out && n > 0, "gad_batch_max: null pointer or empty input (n=%lld)", (long long)n);
    cudaStream_t st = as_stream(stream);
    GAD_CUDA(cudaMemsetAsync(out, 0xff, sizeof(float), st));
    const int64_t blocks = (n + 256 * 8 - 1) / (256 * 8);
    const int grid = (int)(blocks < 4LL * sm_count() ? blocks : 4LL * sm_count());
    k_batch_max<<<grid, 256, 0, st>>>(x, n, reinterpret_cast<unsigned int*>(out));
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" int gad_temp_fold(const float* Mu, const float* temp, int Lw, int CE, float* Mu_eff, void* stream) {
    GAD_CHECK_ARG(Mu && temp && Mu_eff, "gad_temp_fold: null pointer");
    GAD_CHECK_ARG(Lw > 0 && (CE == 2 || CE == 4 || CE == 8), "gad_temp_fold: Lw=%d CE=%d", Lw, CE);
    k_temp_fold<<<1, 256, 0, as_stream(stream)>>>(Mu, temp, Lw, CE * CE + CE, Mu_eff);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" int gad_temp_fold_bwd(const float* gMu, const float* Mu_eff, const float* temp, int Lw, int CE,
                                 float* gMu_base, float* g_temp, void* stream) {
    GAD_CHECK_ARG(gMu && Mu_eff && temp && gMu_base && g_temp, "gad_temp_fold_bwd: null pointer");
    GAD_CHECK_ARG(Lw > 0 && (CE == 2 || CE == 4 || CE == 8), "gad_temp_fold_bwd: Lw=%d CE=%d", Lw, CE);
    k_temp_fold_bwd<<<Lw, TF_THREADS, 0, as_stream(stream)>>>(gMu, Mu_eff, temp, CE * CE + CE, gMu_base, g_temp);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}
