// Global CNN feature extractor of the deformer input (scope row f3): GlobalFeatureExtractorCNN of
// /root/reference/src/feature_extractors.py:6-34, wired at src/GNN.py:242-268 --
//     u <- u / max|u|;  L x [ conv (kernel 3, stride 1, padding 1) + SELU ];  global average pool  ->  [B, C_out]
// on the n x n grid of a mesh's f / uu values (Conv2d) or on the n nodes of a 1-D mesh (Conv1d), one feature
// vector per mesh.  The reference runs it through cuDNN / ATen op by op; here ONE launch per direction, one CTA
// per mesh: the input plane and the activation planes of all L layers live in shared memory (8 channels x 30 x 30
// x 4 layers = 115 KB), weights of the current layer are staged next to them, a thread owns output pixels and
// keeps the C_out accumulators of a pixel in registers.
//   forward : gather the grid through an index map (the canonical-grid reordering of reshape_fd_tensor_to_grid,
//             src/utils_data.py:125-141, fused into the load), layers, fixed-order pooling.
//   backward: forward recomputed into shared memory, then per layer  g_pre = g_act * selu'(act)  (from the stored
//             post-activation: selu' = lambda for act > 0, act + lambda*alpha otherwise), weight gradients one
//             (c_out, c_in, ky, kx) entry per thread summed over the pixels in a fixed order, bias gradients, and
//             the input-plane gradient for the next layer down.  Per-mesh parameter gradients go to a workspace and
//             are summed over the batch in fp64 in a fixed order by a second kernel: no atomics, bit-reproducible.
// The grid values carry no gradient (f / uu are data), as in the reference's use.
#include <stdlib.h>

#include "common.cuh"

namespace gad {
namespace {

constexpr int CNN_MAX_C = 16;
constexpr int CNN_MAX_L = 8;
constexpr int CNN_THREADS = 256;
constexpr float SELU_L = 1.0507009873554804934193349852946f;
constexpr float SELU_A = 1.6732632423543772848170429916717f;

struct CnnArgs {
    const float* u;          // [B, H*W] node values, mesh-major
    const int32_t* gather;   // [H*W] node index of grid cell p (row-major y * W + x), or null = identity
    const float* scale;      // [1] max |u| over the batch (the reference's normalisation)
    const float* w[CNN_MAX_L];
    const float* b[CNN_MAX_L];
    float* out;              // [B, Co]
    const float* g_out;      // [B, Co]             (backward)
    float* g_part;           // [B, n_params]       (backward: per-mesh parameter gradients)
    float* act_global;       // [B, L, Cmax, H*W] or null: activation planes in global memory (L2) when they do not
                             // fit the shared memory next to the other buffers
    float* grad_global;      // [B, 2, Cmax, H*W] or null (backward): the two gradient planes in global memory when
                             // they do not fit the shared memory either
    int B, H, W, Cm, Co, L, KH;
    int n_params;
};

__device__ __forceinline__ float selu(float x) { return SELU_L * (x > 0.f ? x : SELU_A * expm1f(x)); }
__device__ __forceinline__ float selu_grad_from_out(float y) { return y > 0.f ? SELU_L : y + SELU_L * SELU_A; }

__host__ __device__ inline int cnn_cin(const CnnArgs& a, int l) { return l == 0 ? 1 : a.Cm; }
__host__ __device__ inline int cnn_cout(const CnnArgs& a, int l) { return l == a.L - 1 ? a.Co : a.Cm; }
__host__ __device__ inline int cnn_wcount(const CnnArgs& a, int l) { return cnn_cout(a, l) * cnn_cin(a, l) * a.KH * 3; }
__host__ __device__ inline int cnn_param_offset(const CnnArgs& a, int l) {      // flat layout: w_0, b_0, w_1, b_1, ...
    int o = 0;
    for (int k = 0; k < l; ++k) o += cnn_wcount(a, k) + cnn_cout(a, k);
    return o;
}
__host__ __device__ inline int cnn_cmax(const CnnArgs& a) { return a.Cm > a.Co ? a.Cm : a.Co; }

// shared memory: input plane [HW] | L activation planes [Cmax * HW] (unless in global memory) | (backward) two
// gradient planes (unless in global memory) | weights | bias
__host__ __device__ inline size_t cnn_smem_bytes(const CnnArgs& a, bool backward, bool act_in_smem, bool grad_in_smem) {
    const size_t HW = (size_t)a.H * a.W, C = cnn_cmax(a);
    size_t fl = HW + (act_in_smem ? (size_t)a.L * C * HW : 0) + (backward && grad_in_smem ? 2 * C * HW : 0) +
                C * C * a.KH * 3 + C + 64;
    return fl * sizeof(float);
}
__host__ __device__ inline size_t cnn_act_floats(const CnnArgs& a) { return (size_t)a.L * cnn_cmax(a) * a.H * a.W; }
__host__ __device__ inline size_t cnn_grad_floats(const CnnArgs& a) { return (size_t)2 * cnn_cmax(a) * a.H * a.W; }

// layers 0 .. L-1 into the activation planes (all threads; ends with a barrier)
__device__ void cnn_forward_planes(const CnnArgs& a, int mesh, float* in, float* act, float* wsm, float* bsm) {
    const int HW = a.H * a.W, C = cnn_cmax(a), tid = threadIdx.x, nthr = blockDim.x, KH = a.KH;
    const float m = a.scale[0];
    const float* u = a.u + (size_t)mesh * HW;
    for (int p = tid; p < HW; p += nthr) in[p] = u[a.gather ? a.gather[p] : p] / m;
    for (int l = 0; l < a.L; ++l) {
        const int Cin = cnn_cin(a, l), Cout = cnn_cout(a, l), nw = cnn_wcount(a, l);
        __syncthreads();                                   // previous layer's planes complete, weights free
        for (int k = tid; k < nw; k += nthr) wsm[k] = a.w[l][k];
        for (int k = tid; k < Cout; k += nthr) bsm[k] = a.b[l][k];
        __syncthreads();
        const float* src = (l == 0) ? in : act + (size_t)(l - 1) * C * HW;
        float* dst = act + (size_t)l * C * HW;
        for (int p = tid; p < HW; p += nthr) {
            const int y = p / a.W, x = p - y * a.W;
            float acc[CNN_MAX_C];
#pragma unroll
            for (int co = 0; co < CNN_MAX_C; ++co) acc[co] = co < Cout ? bsm[co] : 0.f;
            for (int ci = 0; ci < Cin; ++ci)
                for (int ky = 0; ky < KH; ++ky) {
                    const int yy = y + ky - KH / 2;
                    if (yy < 0 || yy >= a.H) continue;
                    for (int kx = 0; kx < 3; ++kx) {
                        const int xx = x + kx - 1;
                        if (xx < 0 || xx >= a.W) continue;
                        const float v = src[(size_t)ci * HW + yy * a.W + xx];
                        const float* wk = wsm + (ci * KH + ky) * 3 + kx;
#pragma unroll
                        for (int co = 0; co < CNN_MAX_C; ++co)
                            if (co < Cout) acc[co] = fmaf(wk[co * Cin * KH * 3], v, acc[co]);
                    }
                }
#pragma unroll
            for (int co = 0; co < CNN_MAX_C; ++co)
                if (co < Cout) dst[(size_t)co * HW + p] = selu(acc[co]);
        }
    }
    __syncthreads();
}

// fixed-order sum over the pixels of plane[c * HW ..] by one warp (lane-strided partial sums, then a butterfly)
__device__ __forceinline__ float cnn_warp_plane_sum(const float* plane, int HW, int lane) {
    float s = 0.f;
    for (int p = lane; p < HW; p += 32) s += plane[p];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    return s;
}

__global__ void __launch_bounds__(CNN_THREADS) k_cnn_fwd(const CnnArgs a) {
    extern __shared__ __align__(16) float cnn_sm[];
    const int HW = a.H * a.W, C = cnn_cmax(a);
    const int mesh = blockIdx.x;
    float* in = cnn_sm;
    float* act = a.act_global ? a.act_global + (size_t)mesh * cnn_act_floats(a) : in + HW;
    float* wsm = in + HW + (a.act_global ? 0 : cnn_act_floats(a));
    float* bsm = wsm + C * C * a.KH * 3;
    cnn_forward_planes(a, mesh, in, act, wsm, bsm);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const float* last = act + (size_t)(a.L - 1) * C * HW;
    for (int co = warp; co < a.Co; co += nw) {
        const float s = cnn_warp_plane_sum(last + (size_t)co * HW, HW, lane);
        if (lane == 0) a.out[(size_t)mesh * a.Co + co] = s / (float)HW;
    }
}

__global__ void __launch_bounds__(CNN_THREADS) k_cnn_bwd(const CnnArgs a) {
    extern __shared__ __align__(16) float cnn_sm[];
    const int HW = a.H * a.W, C = cnn_cmax(a), KH = a.KH, tid = threadIdx.x, nthr = blockDim.x;
    const int mesh = blockIdx.x;
    float* in = cnn_sm;
    float* act = a.act_global ? a.act_global + (size_t)mesh * cnn_act_floats(a) : in + HW;
    float* gsm = in + HW + (a.act_global ? 0 : cnn_act_floats(a));
    float* gA = a.grad_global ? a.grad_global + (size_t)mesh * cnn_grad_floats(a) : gsm;
    float* gB = gA + (size_t)C * HW;
    float* wsm = a.grad_global ? gsm : gB + (size_t)C * HW;
    float* bsm = wsm + C * C * KH * 3;
    cnn_forward_planes(a, mesh, in, act, wsm, bsm);
    float* gpart = a.g_part + (size_t)mesh * a.n_params;
    // d(mean over pixels) -> last layer's pre-activation gradient
    {
        const float* last = act + (size_t)(a.L - 1) * C * HW;
        const float inv = 1.0f / (float)HW;
        for (int k = tid; k < a.Co * HW; k += nthr) {
            const int co = k / HW;
            gA[k] = a.g_out[(size_t)mesh * a.Co + co] * inv * selu_grad_from_out(last[k]);
        }
    }
    float* gcur = gA;
    float* gnext = gB;
    for (int l = a.L - 1; l >= 0; --l) {
        const int Cin = cnn_cin(a, l), Cout = cnn_cout(a, l), nw = cnn_wcount(a, l), off = cnn_param_offset(a, l);
        __syncthreads();                                   // gcur complete; weights buffer free
        for (int k = tid; k < nw; k += nthr) wsm[k] = a.w[l][k];
        __syncthreads();
        const float* src = (l == 0) ? in : act + (size_t)(l - 1) * C * HW;
        // weight gradients: one entry per thread, pixels in ascending order
        for (int k = tid; k < nw; k += nthr) {
            const int kx = k % 3, ky = (k / 3) % KH, ci = (k / (3 * KH)) % Cin, co = k / (3 * KH * Cin);
            const float* g = gcur + (size_t)co * HW;
            const float* s = src + (size_t)ci * HW;
            float sum = 0.f;
            for (int y = 0; y < a.H; ++y) {
                const int yy = y + ky - KH / 2;
                if (yy < 0 || yy >= a.H) continue;
                const int x0 = (kx == 0) ? 1 : 0, x1 = (kx == 2) ? a.W - 1 : a.W;
                for (int x = x0; x < x1; ++x) sum = fmaf(g[y * a.W + x], s[yy * a.W + x + kx - 1], sum);
            }
            gpart[off + k] = sum;
        }
        // bias gradients: one warp per output channel
        {
            const int warp = tid >> 5, lane = tid & 31, nwp = nthr >> 5;
            for (int co = warp; co < Cout; co += nwp) {
                const float s = cnn_warp_plane_sum(gcur + (size_t)co * HW, HW, lane);
                if (lane == 0) gpart[off + nw + co] = s;
            }
        }
        // gradient of the layer's input planes, times selu' of the layer below
        if (l > 0) {
            const float* below = act + (size_t)(l - 1) * C * HW;
            for (int p = tid; p < HW; p += nthr) {
                const int y = p / a.W, x = p - y * a.W;
                float acc[CNN_MAX_C];
#pragma unroll
                for (int ci = 0; ci < CNN_MAX_C; ++ci) acc[ci] = 0.f;
                for (int co = 0; co < Cout; ++co)
                    for (int ky = 0; ky < KH; ++ky) {
                        const int yy = y - ky + KH / 2;          // output pixel whose tap (ky, kx) reads input (y, x)
                        if (yy < 0 || yy >= a.H) continue;
                        for (int kx = 0; kx < 3; ++kx) {
                            const int xx = x - kx + 1;
                            if (xx < 0 || xx >= a.W) continue;
                            const float g = gcur[(size_t)co * HW + yy * a.W + xx];
                            const float* wk = wsm + (size_t)co * Cin * KH * 3 + ky * 3 + kx;
#pragma unroll
                            for (int ci = 0; ci < CNN_MAX_C; ++ci)
                                if (ci < Cin) acc[ci] = fmaf(wk[ci * KH * 3], g, acc[ci]);
                        }
                    }
#pragma unroll
                for (int ci = 0; ci < CNN_MAX_C; ++ci)
                    if (ci < Cin) gnext[(size_t)ci * HW + p] = acc[ci] * selu_grad_from_out(below[(size_t)ci * HW + p]);
            }
        }
        float* t = gcur;
        gcur = gnext;
        gnext = t;
    }
}

// parameter gradients: sum of the per-mesh parts over the batch, mesh order, fp64
__global__ void k_cnn_reduce(const float* __restrict__ part, int B, int n, float* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    double s = 0.0;
    for (int b = 0; b < B; ++b) s += (double)part[(size_t)b * n + k];
    out[k] = (float)s;
}

int cnn_fill(CnnArgs& a, const float* u, const int32_t* gather, const float* scale, int B, int H, int W, int Cm, int Co,
             int L, const float* const* weights, const float* const* biases) {
    GAD_CHECK_ARG(u && scale && weights && biases && B > 0 && H > 0 && W > 0, "gad_cnn: null argument or empty batch");
    GAD_CHECK_ARG(L >= 2 && L <= CNN_MAX_L && Cm >= 1 && Cm <= CNN_MAX_C && Co >= 1 && Co <= CNN_MAX_C,
                  "gad_cnn: %d layers / %d, %d channels exceed the kernel's limits (%d layers, %d channels)", L, Cm, Co,
                  CNN_MAX_L, CNN_MAX_C);
    a.u = u, a.gather = gather, a.scale = scale;
    a.B = B, a.H = H, a.W = W, a.Cm = Cm, a.Co = Co, a.L = L, a.KH = (H == 1) ? 1 : 3;
    for (int l = 0; l < L; ++l) {
        GAD_CHECK_ARG(weights[l] && biases[l], "gad_cnn: layer %d has no parameters", l);
        a.w[l] = weights[l];
        a.b[l] = biases[l];
    }
    a.n_params = cnn_param_offset(a, L);
    return GAD_OK;
}

}  // namespace
}  // namespace gad

using namespace gad;

extern "C" int64_t gad_cnn_param_count(int H, int Cm, int Co, int L) {
    CnnArgs a{};
    a.H = H, a.Cm = Cm, a.Co = Co, a.L = L, a.KH = (H == 1) ? 1 : 3;
    return cnn_param_offset(a, L);
}

// workspace: [B, n_params] per-mesh parameter gradients (backward), then -- when the activation planes do not fit the
// shared memory -- [B, L, Cmax, H*W] activations, then -- when the backward's two gradient planes do not fit next to the
// input plane either (8 channels: grids beyond about 58 x 58) -- [B, 2, Cmax, H*W] gradient planes.  Activations leave
// shared memory first.  GAD_CNN_GRAD_GLOBAL=1 puts the gradient planes in the workspace whatever fits (read per call;
// the summation order does not depend on where the planes live, so the results are the same bits).
static size_t cnn_plan(CnnArgs& a, bool backward, bool* act_in_smem, bool* grad_in_smem) {
    const char* e = getenv("GAD_CNN_GRAD_GLOBAL");
    const bool force_grad_global = backward && e && e[0] == '1';
    *act_in_smem = !force_grad_global && (int)cnn_smem_bytes(a, backward, true, true) <= smem_optin_bytes();
    *grad_in_smem = !force_grad_global && (int)cnn_smem_bytes(a, backward, *act_in_smem, true) <= smem_optin_bytes();
    return cnn_smem_bytes(a, backward, *act_in_smem, *grad_in_smem);
}

static size_t cnn_grads_bytes(const CnnArgs& a) {
    return ((size_t)a.B * (size_t)gad_cnn_param_count(a.H, a.Cm, a.Co, a.L) * sizeof(float) + 255) & ~(size_t)255;
}

extern "C" size_t gad_cnn_workspace_bytes(int B, int H, int W, int Cm, int Co, int L) {
    CnnArgs a{};
    a.B = B, a.H = H, a.W = W, a.Cm = Cm, a.Co = Co, a.L = L, a.KH = (H == 1) ? 1 : 3;
    bool act_in_smem, grad_in_smem;
    cnn_plan(a, true, &act_in_smem, &grad_in_smem);
    return cnn_grads_bytes(a) + (act_in_smem ? 0 : (size_t)B * cnn_act_floats(a) * sizeof(float)) +
           (grad_in_smem ? 0 : (size_t)B * cnn_grad_floats(a) * sizeof(float)) + 256;
}

extern "C" int gad_cnn_fwd(const float* u, const int32_t* gather, const float* scale, int B, int H, int W, int Cm, int Co,
                           int L, const float* const* weights, const float* const* biases, float* out, void* workspace,
                           size_t workspace_bytes, void* stream) {
    CnnArgs a{};
    int rc = cnn_fill(a, u, gather, scale, B, H, W, Cm, Co, L, weights, biases);
    if (rc) return rc;
    GAD_CHECK_ARG(out, "gad_cnn_fwd: null output");
    a.out = out;
    bool in_smem, unused;
    const size_t bytes = cnn_plan(a, false, &in_smem, &unused);
    GAD_CHECK_ARG((int)bytes <= smem_optin_bytes(), "gad_cnn_fwd: a %d x %d grid with %d channels needs %zu B of shared "
                                                    "memory (> %d)", H, W, cnn_cmax(a), bytes, smem_optin_bytes());
    if (!in_smem) {
        GAD_CHECK_ARG(workspace && workspace_bytes >= (size_t)B * cnn_act_floats(a) * sizeof(float),
                      "gad_cnn_fwd: the activation planes need a workspace of gad_cnn_workspace_bytes");
        a.act_global = reinterpret_cast<float*>(workspace);
    }
    GAD_CUDA(cudaFuncSetAttribute(k_cnn_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    k_cnn_fwd<<<B, CNN_THREADS, bytes, as_stream(stream)>>>(a);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" int gad_cnn_bwd(const float* u, const int32_t* gather, const float* scale, int B, int H, int W, int Cm, int Co,
                           int L, const float* const* weights, const float* const* biases, const float* g_out,
                           float* g_params, void* workspace, size_t workspace_bytes, void* stream) {
    CnnArgs a{};
    int rc = cnn_fill(a, u, gather, scale, B, H, W, Cm, Co, L, weights, biases);
    if (rc) return rc;
    GAD_CHECK_ARG(g_out && g_params && workspace, "gad_cnn_bwd: null argument");
    GAD_CHECK_ARG(workspace_bytes >= gad_cnn_workspace_bytes(B, H, W, Cm, Co, L), "gad_cnn_bwd: workspace too small");
    a.g_out = g_out;
    a.g_part = reinterpret_cast<float*>(workspace);
    bool act_in_smem, grad_in_smem;
    const size_t bytes = cnn_plan(a, true, &act_in_smem, &grad_in_smem);
    GAD_CHECK_ARG((int)bytes <= smem_optin_bytes(), "gad_cnn_bwd: a %d x %d grid with %d channels needs %zu B of shared "
                                                    "memory (> %d)", H, W, cnn_cmax(a), bytes, smem_optin_bytes());
    char* next = reinterpret_cast<char*>(workspace) + cnn_grads_bytes(a);
    if (!act_in_smem) {
        a.act_global = reinterpret_cast<float*>(next);
        next += (size_t)B * cnn_act_floats(a) * sizeof(float);
    }
    if (!grad_in_smem) a.grad_global = reinterpret_cast<float*>(next);
    GAD_CUDA(cudaFuncSetAttribute(k_cnn_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    cudaStream_t st = as_stream(stream);
    k_cnn_bwd<<<B, CNN_THREADS, bytes, st>>>(a);
    GAD_LAUNCH_CHECK();
    k_cnn_reduce<<<(a.n_params + 127) / 128, 128, 0, st>>>(a.g_part, B, a.n_params, g_params);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}
