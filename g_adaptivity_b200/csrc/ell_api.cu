// Host side of the mesh-resident ELL kernels (ell_kernels.cuh): the ELL topology builder, the
// launch planner (threads per CTA, ELL rows in shared memory or streamed from L2), the fixed-order
// reduction of the per-tile partials, and the C-ABI entry points of include/gadapt.h.
#include <stdlib.h>

#include "ell_kernels.cuh"

namespace gad {
namespace ell {

GAD_ELL_DECLARE(2, 2)
GAD_ELL_DECLARE(2, 3)
GAD_ELL_DECLARE(2, 6)
GAD_ELL_DECLARE(2, 7)
GAD_ELL_DECLARE(4, 2)
GAD_ELL_DECLARE(4, 3)
GAD_ELL_DECLARE(4, 6)
GAD_ELL_DECLARE(4, 7)

namespace {

// ---- ELL rows from the CSR / CSC walk arrays -----------------------------------------------
// One CTA per tile.  ell[i] = { (row_q - n0) * ROWBYTES as uint16 for q < 7 ; 7-bit validity mask }.
// Slot choice: the first W distinct neighbour offsets (j - i) met in the tile define the canonical
// slots; a neighbour goes to the slot of its offset when that slot is free (else to any free slot),
// and an empty slot is padded with the row the canonical offset points at (clamped into the tile).
// On a structured mesh slot q then means "the same direction" for every node, boundary nodes
// included, so the q-th gather of consecutive lanes reads consecutive rows: no bank conflicts.
// Any assignment is CORRECT (the kernels mask by the validity bits); this one is merely fast.
__global__ void k_build_ell(const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                            const int32_t* __restrict__ tile_ptr, int T, int rowbytes, int W, uint4* __restrict__ ell,
                            int32_t* __restrict__ bad) {
    const int t = blockIdx.x;
    if (t >= T) return;
    __shared__ int tab[ELL_SLOTS];
    __shared__ int ntab_s;
    const int n0 = tile_ptr[t], n1 = tile_ptr[t + 1];
    if (threadIdx.x == 0) {
        int nt = 0;
        for (int i = n0; i < n1 && nt < W; ++i)
            for (int e = ptr[i]; e < ptr[i + 1] && nt < W; ++e) {
                const int d = idx[e] - i;
                bool seen = false;
                for (int q = 0; q < nt; ++q) seen |= (tab[q] == d);
                if (!seen) tab[nt++] = d;
            }
        ntab_s = nt;
    }
    __syncthreads();
    const int ntab = ntab_s;
    for (int i = n0 + threadIdx.x; i < n1; i += blockDim.x) {
        const int b = ptr[i], e = ptr[i + 1];
        const int deg = e - b;
        int slot[ELL_SLOTS];
        for (int q = 0; q < ELL_SLOTS; ++q) slot[q] = -1;
        bool ok = (deg <= W);
        unsigned placed = 0;
        if (ok) {
            for (int k = 0; k < deg; ++k) {           // canonical slot of the neighbour's offset
                const int j = idx[b + k];
                if (j < n0 || j >= n1) ok = false;
                for (int q = 0; q < ntab; ++q)
                    if (!(placed >> k & 1u) && slot[q] < 0 && tab[q] == j - i) {
                        slot[q] = j;
                        placed |= 1u << k;
                    }
            }
            for (int k = 0; k < deg; ++k) {           // leftovers: any free slot
                if (placed >> k & 1u) continue;
                for (int q = 0; q < W; ++q)
                    if (slot[q] < 0) {
                        slot[q] = idx[b + k];
                        placed |= 1u << k;
                        break;
                    }
            }
        }
        uint32_t h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        uint32_t mask = 0;
        for (int q = 0; q < ELL_SLOTS; ++q) {
            int j;
            if (ok && slot[q] >= 0) {
                j = slot[q];
                mask |= 1u << q;
            } else {
                j = i + ((q < ntab) ? tab[q] : 0);    // padding: a valid row, masked out by the kernels
                j = j < n0 ? n0 : (j >= n1 ? n1 - 1 : j);
            }
            const long long off = (long long)(j - n0) * rowbytes;
            if (off > 0xffff) ok = false;
            h[q] = (uint32_t)(off & 0xffff);
        }
        if (!ok) {
            atomicAdd(bad, 1);
            for (int q = 0; q < 8; ++q) h[q] = 0;
            mask = 0;
        }
        h[7] = mask;
        ell[i] = make_uint4(h[0] | (h[1] << 16), h[2] | (h[3] << 16), h[4] | (h[5] << 16), h[6] | (h[7] << 16));
    }
}

// ---- fixed-order reduction of the per-tile partials -------------------------------------------
// One warp per output column: columns [0, slots*nacc) are (G_M, G_u[, g_tau]) per weight slot,
// then L step-size columns (shared weights) and one loss column.
__global__ void k_ell_reduce(const float* __restrict__ partials, int T, int slots, int nacc, int musz,
                             float* __restrict__ gMu, const float* __restrict__ tau_partials, int L,
                             float* __restrict__ g_tau, const float* __restrict__ loss_partials, float loss_scale,
                             float* __restrict__ loss) {
    tail::reduce_partials(partials, T, slots, nacc, musz, gMu, tau_partials, L, g_tau, loss_partials, loss_scale, loss,
                          blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), gridDim.x * (blockDim.x >> 5));
}

// instantiated slot counts: 2, 3, 6, 7
int slots_for(int max_deg) { return max_deg <= 2 ? 2 : (max_deg <= 3 ? 3 : (max_deg <= 6 ? 6 : 7)); }

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

struct Plan {
    int w;        // instantiated slot count (2, 3, 6, 7)
    int ells;     // ELL rows staged in shared memory
    int threads;
};

// Per-SM shared memory: 228 KB minus 1 KB reserved per resident CTA.
constexpr size_t SMEM_PER_SM = 233472;

int make_plan(int CE, int kind, int max_tile_nodes, int max_deg, Plan* p) {
    GAD_CHECK_ARG(CE == 2 || CE == 4, "ELL kernels are instantiated for CE = 2 and 4 (got %d)", CE);
    GAD_CHECK_ARG(max_deg >= 0 && max_deg <= ELL_SLOTS, "ELL kernels need degree <= %d (got %d)", ELL_SLOTS, max_deg);
    GAD_CHECK_ARG(max_tile_nodes > 0 && (long long)max_tile_nodes * CE * 4 <= 0x10000,
                  "ELL kernels: tile of %d nodes exceeds the 16-bit row offsets", max_tile_nodes);
    p->w = slots_for(max_deg);
    const int nw = GAD_ELL_MAXT / 32;
    const size_t with = make_layout(CE, kind, max_tile_nodes, true, nw).total + 1024;
    const size_t without = make_layout(CE, kind, max_tile_nodes, false, nw).total + 1024;
    const size_t optin = (size_t)smem_optin_bytes() + 1024;
    int ells;
    if (2 * with <= SMEM_PER_SM) ells = 1;                 // two CTAs per SM either way
    else if (2 * without <= SMEM_PER_SM) ells = 0;         // keep the second CTA
    else if (with <= optin) ells = 1;
    else if (without <= optin) ells = 0;
    else {
        set_error("ELL kernels: a tile of %d nodes needs %zu B of shared memory (> %zu)", max_tile_nodes, without, optin);
        return GAD_ERR_UNSUPPORTED;
    }
    ells = env_int("GAD_ELL_SMEM", ells);
    p->ells = ells ? 1 : 0;
    const size_t bytes = p->ells ? with : without;
    const bool two = 2 * bytes <= SMEM_PER_SM;
    int target = env_int("GAD_ELL_THREADS", two ? GAD_ELL_MAXT / 2 : GAD_ELL_MAXT);
    if (target > GAD_ELL_MAXT) target = GAD_ELL_MAXT;
    if (target < 32) target = 32;
    const int rounds = (max_tile_nodes + target - 1) / target;
    int th = (max_tile_nodes + rounds - 1) / rounds;
    th = ((th + 31) / 32) * 32;
    if (th < 64) th = 64;
    if (th > GAD_ELL_MAXT) th = GAD_ELL_MAXT;
    p->threads = th;
    return GAD_OK;
}

int dispatch(int CE, const Plan& p, int which, const Args& a, int method, cudaStream_t st) {
#define GAD_ELL_CASE(CE_, W_) \
    if (CE == CE_ && p.w == W_) return ell_launch_c##CE_##w##W_(which, a, method, p.ells, p.threads, st)
    GAD_ELL_CASE(2, 2);
    GAD_ELL_CASE(2, 3);
    GAD_ELL_CASE(2, 6);
    GAD_ELL_CASE(2, 7);
    GAD_ELL_CASE(4, 2);
    GAD_ELL_CASE(4, 3);
    GAD_ELL_CASE(4, 6);
    GAD_ELL_CASE(4, 7);
#undef GAD_ELL_CASE
    set_error("ELL kernels: no instantiation for CE=%d W=%d", CE, p.w);
    return GAD_ERR_UNSUPPORTED;
}

size_t ws_floats(int CE, int T, int L) {
    const int NACC = CE * CE + CE + 1;
    return (size_t)T * L * NACC + (size_t)T * L + (size_t)T + 64;
}

int reduce_partials(int CE, int T, int Lw, int L, float* ws, float* gMu, float* g_tau, float loss_scale, float* loss,
                    cudaStream_t st) {
    const int NACC = CE * CE + CE + 1, MUSZ = CE * CE + CE;
    const int slots = Lw > 1 ? L : 1;
    float* partials = ws;
    float* tau_partials = (g_tau && Lw == 1) ? ws + (size_t)T * L * NACC : nullptr;
    float* loss_partials = loss ? ws + (size_t)T * L * NACC + (size_t)T * L : nullptr;
    const int ncol = slots * NACC + L + 1;
    k_ell_reduce<<<(ncol + 7) / 8, 256, 0, st>>>(partials, T, slots, NACC, MUSZ, gMu, tau_partials, L, g_tau,
                                                 loss_partials, loss_scale, loss);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

}  // namespace
}  // namespace ell
}  // namespace gad

using namespace gad;
using namespace gad::ell;

// tile_ptr == NULL: shared-topology batch of equal tiles (include/gadapt.h) -- the tile count must match
#define GAD_UNIFORM_TILES_OK(who)                                                                                  \
    GAD_CHECK_ARG(tile_ptr || (max_tile_nodes > 0 && (int64_t)T == (N + max_tile_nodes - 1) / max_tile_nodes),     \
                  who ": tile_ptr == NULL means T = ceil(N / max_tile_nodes) equal tiles (N=%lld T=%d tile=%d)",    \
                  (long long)N, T, max_tile_nodes)

extern "C" int gad_graph_build_ell(const int32_t* ptr, const int32_t* idx, int64_t N, const int32_t* tile_ptr, int T,
                                   int CE, int max_deg, void* ell_rows, int32_t* info, void* stream) {
    GAD_CHECK_ARG(ptr && idx && tile_ptr && ell_rows && info && N > 0 && T > 0, "gad_graph_build_ell: bad arguments");
    GAD_CHECK_ARG(CE == 2 || CE == 4, "gad_graph_build_ell: CE must be 2 or 4 (got %d)", CE);
    GAD_CHECK_ARG(max_deg >= 0 && max_deg <= ELL_SLOTS, "gad_graph_build_ell: max_deg=%d exceeds %d slots", max_deg,
                  ELL_SLOTS);
    k_build_ell<<<T, 128, 0, as_stream(stream)>>>(ptr, idx, tile_ptr, T, CE * 4, slots_for(max_deg),
                                                 reinterpret_cast<uint4*>(ell_rows), info + GAD_INFO_ELL_BAD);
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}

extern "C" int gad_ell_supported(int CE, int max_tile_nodes, int max_deg, int train) {
    Plan p;
    if (CE != 2 && CE != 4) return 0;
    if (max_deg > ELL_SLOTS || max_tile_nodes <= 0 || (long long)max_tile_nodes * CE * 4 > 0x10000) return 0;
    if (make_plan(CE, KIND_FWD_RK4, max_tile_nodes, max_deg, &p) != GAD_OK) return 0;
    if (train && make_plan(CE, KIND_BWD, max_tile_nodes, max_deg, &p) != GAD_OK) return 0;
    return 1;
}

extern "C" size_t gad_ell_workspace_bytes(int CE, int T, int L) { return ws_floats(CE, T > 0 ? T : 1, L) * sizeof(float); }

extern "C" int gad_deform_fwd_ell(const void* ell_in, int64_t N, const int32_t* tile_ptr, int T, int max_tile_nodes,
                                  int max_deg, const float* x0, int dim, int CE, const float* Mu, int Lw,
                                  const float* tau, int L, int method, float* x_phys, float* states, void* stream) {
    GAD_CHECK_ARG(ell_in && x0 && Mu && tau && x_phys, "gad_deform_fwd_ell: null pointer");
    GAD_UNIFORM_TILES_OK("gad_deform_fwd_ell");
    GAD_CHECK_ARG(N > 0 && T > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L),
                  "gad_deform_fwd_ell: N=%lld T=%d L=%d dim=%d CE=%d Lw=%d", (long long)N, T, L, dim, CE, Lw);
    GAD_CHECK_ARG(method == GAD_METHOD_EULER || method == GAD_METHOD_RK4, "gad_deform_fwd_ell: unknown method %d", method);
    GAD_CHECK_ARG(!states || states == x0, "gad_deform_fwd_ell: when states is given, x0 must alias states[0]");
    Plan p;
    int rc = make_plan(CE, method == GAD_METHOD_RK4 ? KIND_FWD_RK4 : KIND_FWD, max_tile_nodes, max_deg, &p);
    if (rc) return rc;
    Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(ell_in);
    a.tile_ptr = tile_ptr;
    a.T = T;
    a.cap_nodes = max_tile_nodes;
    a.N = N;
    a.Mu = Mu;
    a.tau = tau;
    a.Lw = Lw;
    a.L = L;
    a.dim = dim;
    a.x0 = x0;
    a.x_phys = x_phys;
    a.states = states;
    return dispatch(CE, p, 0, a, method, as_stream(stream));
}

extern "C" int gad_deform_fwd_ell_raw(const void* ell_in, int64_t N, const int32_t* tile_ptr, int T,
                                      int max_tile_nodes, int max_deg, const float* x_comp, const float* f,
                                      const float* uu, const float* f_scale, const float* uu_scale, int dim, int CE,
                                      const float* Mu, const float* du, int Lw, const float* tau, int L, int method,
                                      float* x_phys, float* states, void* stream) {
    GAD_CHECK_ARG(ell_in && x_comp && Mu && tau && x_phys, "gad_deform_fwd_ell_raw: null pointer");
    GAD_UNIFORM_TILES_OK("gad_deform_fwd_ell_raw");
    GAD_CHECK_ARG(N > 0 && T > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L),
                  "gad_deform_fwd_ell_raw: N=%lld T=%d L=%d dim=%d CE=%d Lw=%d", (long long)N, T, L, dim, CE, Lw);
    GAD_CHECK_ARG(dim + (f ? 1 : 0) + (uu ? 1 : 0) <= CE, "gad_deform_fwd_ell_raw: %d input features exceed CE=%d",
                  dim + (f ? 1 : 0) + (uu ? 1 : 0), CE);
    GAD_CHECK_ARG(method == GAD_METHOD_EULER || method == GAD_METHOD_RK4, "gad_deform_fwd_ell_raw: unknown method %d",
                  method);
    Plan p;
    int rc = make_plan(CE, method == GAD_METHOD_RK4 ? KIND_FWD_RK4 : KIND_FWD, max_tile_nodes, max_deg, &p);
    if (rc) return rc;
    Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(ell_in);
    a.tile_ptr = tile_ptr;
    a.T = T;
    a.cap_nodes = max_tile_nodes;
    a.N = N;
    a.Mu = Mu;
    a.tau = tau;
    a.Lw = Lw;
    a.L = L;
    a.dim = dim;
    a.x0 = nullptr;          // selects the fused feature assembly
    a.du = du;
    a.x_comp = x_comp;
    a.f = f;
    a.uu = uu;
    a.f_scale = f_scale;
    a.uu_scale = uu_scale;
    a.x_phys = x_phys;
    a.states = states;
    return dispatch(CE, p, 0, a, method, as_stream(stream));
}

extern "C" int gad_deform_bwd_ell(const void* ell_in, const void* ell_out, int64_t N, const int32_t* tile_ptr, int T,
                                  int max_tile_nodes, int max_deg, const float* states, const float* g_xphys, int dim,
                                  int CE, const float* Mu, const float* du, int Lw, const float* tau, int L, float* gMu,
                                  float* g_tau, float* g_x0, void* workspace, size_t workspace_bytes, void* stream) {
    GAD_CHECK_ARG(ell_in && ell_out && states && g_xphys && Mu && tau && gMu && workspace,
                  "gad_deform_bwd_ell: null pointer");
    GAD_UNIFORM_TILES_OK("gad_deform_bwd_ell");
    GAD_CHECK_ARG(N > 0 && T > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L),
                  "gad_deform_bwd_ell: N=%lld T=%d L=%d dim=%d CE=%d Lw=%d", (long long)N, T, L, dim, CE, Lw);
    GAD_CHECK_ARG(workspace_bytes >= ws_floats(CE, T, L) * sizeof(float), "gad_deform_bwd_ell: workspace too small");
    Plan p;
    int rc = make_plan(CE, KIND_BWD, max_tile_nodes, max_deg, &p);
    if (rc) return rc;
    const int NACC = CE * CE + CE + 1;
    float* ws = reinterpret_cast<float*>(workspace);
    Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(ell_in);
    a.ell_out = reinterpret_cast<const uint4*>(ell_out);
    a.tile_ptr = tile_ptr;
    a.T = T;
    a.cap_nodes = max_tile_nodes;
    a.N = N;
    a.Mu = Mu;
    a.tau = tau;
    a.Lw = Lw;
    a.L = L;
    a.dim = dim;
    a.states = const_cast<float*>(states);
    a.g_xphys = g_xphys;
    a.du = du;
    a.partials = ws;
    a.tau_partials = (g_tau && Lw == 1) ? ws + (size_t)T * L * NACC : nullptr;
    a.g_x0 = g_x0;
    cudaStream_t st = as_stream(stream);
    if ((rc = dispatch(CE, p, 1, a, GAD_METHOD_EULER, st))) return rc;
    return reduce_partials(CE, T, Lw, L, ws, gMu, g_tau, 0.f, nullptr, st);
}

extern "C" int gad_deform_bwd_ell_rk4(const void* ell_in, const void* ell_out, int64_t N, const int32_t* tile_ptr, int T,
                                      int max_tile_nodes, int max_deg, const float* states, const float* g_xphys, int dim,
                                      int CE, const float* Mu, const float* du, int Lw, const float* tau, int L, float* gMu,
                                      float* g_x0, void* workspace, size_t workspace_bytes, void* stream) {
    GAD_CHECK_ARG(ell_in && ell_out && states && g_xphys && Mu && tau && gMu && workspace, "gad_deform_bwd_ell_rk4: null pointer");
    GAD_UNIFORM_TILES_OK("gad_deform_bwd_ell_rk4");
    GAD_CHECK_ARG(N > 0 && T > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L),
                  "gad_deform_bwd_ell_rk4: N=%lld T=%d L=%d dim=%d CE=%d Lw=%d", (long long)N, T, L, dim, CE, Lw);
    GAD_CHECK_ARG(workspace_bytes >= ws_floats(CE, T, L) * sizeof(float), "gad_deform_bwd_ell_rk4: workspace too small");
    Plan p;
    int rc = make_plan(CE, KIND_BWD_RK4, max_tile_nodes, max_deg, &p);
    if (rc) return rc;
    float* ws = reinterpret_cast<float*>(workspace);
    Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(ell_in);
    a.ell_out = reinterpret_cast<const uint4*>(ell_out);
    a.tile_ptr = tile_ptr;
    a.T = T;
    a.cap_nodes = max_tile_nodes;
    a.N = N;
    a.Mu = Mu;
    a.tau = tau;
    a.Lw = Lw;
    a.L = L;
    a.dim = dim;
    a.states = const_cast<float*>(states);
    a.g_xphys = g_xphys;
    a.du = du;
    a.partials = ws;
    a.tau_partials = nullptr;
    a.g_x0 = g_x0;
    cudaStream_t st = as_stream(stream);
    if ((rc = dispatch(CE, p, 3, a, GAD_METHOD_RK4, st))) return rc;
    return reduce_partials(CE, T, Lw, L, ws, gMu, nullptr, 0.f, nullptr, st);
}

extern "C" int gad_ell_rk4_bwd_supported(int CE, int max_tile_nodes, int max_deg) {
    Plan p;
    if (CE != 2 && CE != 4) return 0;
    if (max_deg > ELL_SLOTS || max_tile_nodes <= 0 || (long long)max_tile_nodes * CE * 4 > 0x10000) return 0;
    return make_plan(CE, KIND_BWD_RK4, max_tile_nodes, max_deg, &p) == GAD_OK ? 1 : 0;
}

extern "C" int gad_deform_train_ell(const void* ell_in, const void* ell_out, int64_t N, const int32_t* tile_ptr, int T,
                                    int max_tile_nodes, int max_deg, const float* x_comp, const float* f,
                                    const float* uu, const float* f_scale, const float* uu_scale, const float* target,
                                    int dim, int CE, const float* Mu, int Lw, const float* tau, int L, int loss_kind,
                                    float grad_scale, float loss_scale, float* states, float* gMu, float* g_tau,
                                    float* loss, float* x_phys, void* workspace, size_t workspace_bytes, void* stream) {
    GAD_CHECK_ARG(ell_in && ell_out && x_comp && target && Mu && tau && states && gMu && loss && workspace,
                  "gad_deform_train_ell: null pointer");
    GAD_UNIFORM_TILES_OK("gad_deform_train_ell");
    GAD_CHECK_ARG(N > 0 && T > 0 && L > 0 && dim >= 1 && dim <= CE && (Lw == 1 || Lw == L),
                  "gad_deform_train_ell: N=%lld T=%d L=%d dim=%d CE=%d Lw=%d", (long long)N, T, L, dim, CE, Lw);
    GAD_CHECK_ARG(dim + (f ? 1 : 0) + (uu ? 1 : 0) <= CE, "gad_deform_train_ell: %d input features exceed CE=%d",
                  dim + (f ? 1 : 0) + (uu ? 1 : 0), CE);
    GAD_CHECK_ARG(loss_kind == 0 || loss_kind == 1, "gad_deform_train_ell: unknown loss kind %d", loss_kind);
    GAD_CHECK_ARG(workspace_bytes >= ws_floats(CE, T, L) * sizeof(float), "gad_deform_train_ell: workspace too small");
    Plan p;
    int rc = make_plan(CE, KIND_BWD, max_tile_nodes, max_deg, &p);
    if (rc) return rc;
    const int NACC = CE * CE + CE + 1;
    float* ws = reinterpret_cast<float*>(workspace);
    Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(ell_in);
    a.ell_out = reinterpret_cast<const uint4*>(ell_out);
    a.tile_ptr = tile_ptr;
    a.T = T;
    a.cap_nodes = max_tile_nodes;
    a.N = N;
    a.Mu = Mu;
    a.tau = tau;
    a.Lw = Lw;
    a.L = L;
    a.dim = dim;
    a.x_phys = x_phys;
    a.states = states;
    a.partials = ws;
    a.tau_partials = (g_tau && Lw == 1) ? ws + (size_t)T * L * NACC : nullptr;
    a.g_x0 = nullptr;
    a.x_comp = x_comp;
    a.f = f;
    a.uu = uu;
    a.f_scale = f_scale;
    a.uu_scale = uu_scale;
    a.target = target;
    a.loss_kind = loss_kind;
    a.grad_scale = grad_scale;
    a.loss_partials = ws + (size_t)T * L * NACC + (size_t)T * L;
    cudaStream_t st = as_stream(stream);
    if ((rc = dispatch(CE, p, 2, a, GAD_METHOD_EULER, st))) return rc;
    return reduce_partials(CE, T, Lw, L, ws, gMu, g_tau, loss_scale, loss, st);
}

// One training step of gad_train_step_ell / gad_train_step_ell_rk4 (`who` names the entry point in errors).
static int train_step(const gad_train_desc* d, int method, const char* who, void* stream) {
    GAD_CHECK_ARG(d, "%s: null descriptor", who);
    GAD_CHECK_ARG(d->ell_in && d->ell_out && d->x_comp && d->target && d->Mu && d->tau && d->states &&
                      d->gMu && d->loss && d->workspace && d->counter,
                  "%s: null pointer", who);
    GAD_CHECK_ARG(d->tile_ptr || (d->max_tile_nodes > 0 &&
                                  (int64_t)d->T == (d->N + d->max_tile_nodes - 1) / d->max_tile_nodes),
                  "%s: tile_ptr == NULL means T = ceil(N / max_tile_nodes) equal tiles (N=%lld T=%d tile=%d)", who,
                  (long long)d->N, d->T, d->max_tile_nodes);
    GAD_CHECK_ARG(d->N > 0 && d->T > 0 && d->L > 0 && d->dim >= 1 && d->dim <= d->CE && (d->Lw == 1 || d->Lw == d->L),
                  "%s: N=%lld T=%d L=%d dim=%d CE=%d Lw=%d", who, (long long)d->N, d->T, d->L, d->dim, d->CE, d->Lw);
    GAD_CHECK_ARG(d->dim + (d->f ? 1 : 0) + (d->uu ? 1 : 0) <= d->CE, "%s: input features exceed CE=%d", who, d->CE);
    GAD_CHECK_ARG(d->loss_kind == 0 || d->loss_kind == 1, "%s: unknown loss kind %d", who, d->loss_kind);
    GAD_CHECK_ARG(d->tail == 1 || d->tail == 2, "%s: tail must be 1 or 2 (got %d)", who, d->tail);
    GAD_CHECK_ARG(d->Wq && d->bq && d->Wk && d->gWq && d->gbq && d->gWk && d->gbk && d->C > 0,
                  "%s: the tail needs the Linear parameters and their gradient buffers", who);
    GAD_CHECK_ARG(d->tail < 2 || (d->params && d->grads && d->exp_avg && d->exp_avg_sq && d->step && d->n_params > 0),
                  "%s: tail == 2 needs the flat parameter vector and the Adam state", who);
    GAD_CHECK_ARG(d->workspace_bytes >= ws_floats(d->CE, d->T, d->L) * sizeof(float), "%s: workspace too small", who);
    GAD_CHECK_ARG(method == GAD_METHOD_EULER || d->g_tau == nullptr,
                  "%s: the step sizes get no gradient through RK4 (g_tau must be NULL)", who);
    const int kind = method == GAD_METHOD_RK4 ? KIND_TRAIN_RK4 : KIND_BWD;
    Plan p;
    int rc = make_plan(d->CE, kind, d->max_tile_nodes, d->max_deg, &p);
    if (rc) return rc;
    const int NACC = d->CE * d->CE + d->CE + 1;
    float* ws = reinterpret_cast<float*>(d->workspace);
    Args a{};
    a.ell_in = reinterpret_cast<const uint4*>(d->ell_in);
    a.ell_out = reinterpret_cast<const uint4*>(d->ell_out);
    a.tile_ptr = d->tile_ptr;
    a.T = d->T;
    a.cap_nodes = d->max_tile_nodes;
    a.N = d->N;
    a.Mu = d->Mu;
    a.tau = d->tau;
    a.Lw = d->Lw;
    a.L = d->L;
    a.dim = d->dim;
    a.x_phys = d->x_phys;
    a.states = d->states;
    a.partials = ws;
    a.tau_partials = (d->g_tau && d->Lw == 1) ? ws + (size_t)d->T * d->L * NACC : nullptr;
    a.x_comp = d->x_comp;
    a.f = d->f;
    a.uu = d->uu;
    a.f_scale = d->f_scale;
    a.uu_scale = d->uu_scale;
    a.target = d->target;
    a.loss_kind = d->loss_kind;
    a.grad_scale = d->grad_scale;
    a.loss_partials = ws + (size_t)d->T * d->L * NACC + (size_t)d->T * d->L;
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
    cudaStream_t st = as_stream(stream);
    // The in-kernel tail keeps mirrors of the flat parameter / gradient vectors in shared memory: it
    // needs Wq / bq / Wk to be views of `params` (tail 2) and its scratch plan to fit the CTA.
    auto within = [](const float* q, const float* base, long long n) { return q >= base && q < base + n; };
    const long long np = d->tail >= 2 ? d->n_params : 0;
    const Layout lay = make_layout(d->CE, kind, d->max_tile_nodes, p.ells != 0, (p.threads + 31) / 32);
    const TailPlan tplan = plan_tail(d->CE, d->Lw, d->L, d->C, a.tau_partials && a.g_tau, true, np, d->T, (p.threads + 31) / 32,
                                     lay.bar);
    bool fused_tail = tplan.ok;
    if (d->world > 1 && d->peers)   // received peer gradients [world][n_params] sit in the tail's staging area
        fused_tail = fused_tail && (size_t)d->world * (size_t)np * sizeof(float) <= tplan.stage_bytes;
    if (d->tail >= 2) {
        const float* views[] = {d->Wq, d->bq, d->Wk};
        const float* gviews[] = {d->gWq, d->gbq, d->gWk, d->gbk};
        for (const float* v : views) fused_tail = fused_tail && within(v, d->params, np);
        for (const float* v : gviews) fused_tail = fused_tail && within(v, d->grads, np);
        if (d->g_tau) fused_tail = fused_tail && within(d->g_tau, d->grads, np);
    }
    const bool exchange = d->world > 1 && d->peers;
    if (exchange) {
        GAD_CHECK_ARG(d->tail == 2 && d->peer_seq && d->rank >= 0 && d->rank < d->world && d->world <= GAD_MAX_PEERS,
                      "%s: the peer exchange needs tail == 2, a sequence counter and rank < world <= %d", who,
                      GAD_MAX_PEERS);
        GAD_CHECK_ARG(fused_tail, "%s: the peer exchange needs the in-kernel tail (flat parameter views, scratch of %u B)",
                      who, lay.bar);
    }
    if (fused_tail) return dispatch(d->CE, p, 2, a, method, st);
    // generic path: the same step as separate launches
    a.tail = 0;
    a.pdl = 0;
    if ((rc = dispatch(d->CE, p, 2, a, method, st))) return rc;
    if ((rc = reduce_partials(d->CE, d->T, d->Lw, d->L, ws, d->gMu, d->g_tau, d->loss_scale, d->loss, st))) return rc;
    if ((rc = gad_weight_grads(d->Wq, d->bq, d->Wk, d->gMu, d->Lw, d->C, d->CE, d->inv_temp, d->gWq, d->gbq, d->gWk, d->gbk,
                               stream)))
        return rc;
    if (d->tail >= 2) {
        if ((rc = gad_adam_step(d->params, d->grads, d->exp_avg, d->exp_avg_sq, d->n_params, d->lr, d->beta1, d->beta2,
                                d->eps, d->weight_decay, d->adam_grad_scale, d->step, stream)))
            return rc;
        if ((rc = gad_prepare_weights(d->Wq, d->bq, d->Wk, d->Lw, d->C, d->CE, d->inv_temp, d->Mu, stream))) return rc;
    }
    return GAD_OK;
}

extern "C" int gad_train_step_ell(const gad_train_desc* d, void* stream) {
    return train_step(d, GAD_METHOD_EULER, "gad_train_step_ell", stream);
}

extern "C" int gad_train_step_ell_rk4(const gad_train_desc* d, void* stream) {
    return train_step(d, GAD_METHOD_RK4, "gad_train_step_ell_rk4", stream);
}

extern "C" int gad_ell_rk4_train_supported(int CE, int max_tile_nodes, int max_deg) {
    Plan p;
    if (CE != 2 && CE != 4) return 0;
    if (max_deg > ELL_SLOTS || max_tile_nodes <= 0 || (long long)max_tile_nodes * CE * 4 > 0x10000) return 0;
    return make_plan(CE, KIND_TRAIN_RK4, max_tile_nodes, max_deg, &p) == GAD_OK ? 1 : 0;
}
