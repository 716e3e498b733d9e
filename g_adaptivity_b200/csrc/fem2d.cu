// Batched differentiable 2-D P1 finite-element solve behind loss_type = 'pde_loss' on 2-D meshes (scope row f1,
// second half): torch_FEM_2D of /root/reference/firedrake_difFEM/difFEM_2d.py:345-372, which the reference runs per
// mesh in a Python loop (src/GNN.py:327-335), as one CTA per mesh over a topology shared by the batch.
//
// Its arithmetic (fem2d_math.cuh) and phase order are checked on the CPU against the reference's fixtures
// (oracle/fem2d_host.cpp, tests/test_fem2d_oracle.py), the kernels below also run on the CPU under a
// thread-per-CUDA-thread emulation (oracle/fem2d_emu.cpp: FEM2D_EMULATE), and on the B200 they match the fixtures to
// 4e-6 / 1.2e-5 (forward / gradient; tests/test_fem2d_gpu.py).  GNN.forward routes 2-D pde_loss here (GNN._pde_tail_2d).
//
// Phases (forward): coordinates + cells -> shared memory; load vector (Simpson cubature per interior node, one warp
// per node; Dirichlet values); the interior stiffness matrix as padded rows in shared memory (<= D + 2 entries per
// node: uint16 column, fp64 coefficient = sum of the fp32 local entries, column-major so that consecutive threads
// read consecutive words); conjugate gradients on the SPD interior system in fp64 -- one thread per row, the p.Ap
// and r.r partial sums fused into the row loops, three barriers per iteration; interpolation on the evaluation
// points through a uniform bin table over the mesh's bounding box (cells binned by their inflated bounding boxes;
// a point tests the cells of its bin only, and its hits are sorted by cell id, so the result is that of the
// reference's scan over all cells in ascending order).
// Backward: g_u by fp64 shared-memory accumulation, second CG solve for the adjoint, three gradient terms
// (matrix, load vector, interpolation) accumulated per vertex in shared memory, one store per vertex.
// Round 1 (one thread per CG row gathering through the global star tables, all-cells point location) took 36 ms
// for 256 meshes of 30x30, forward + backward.
#ifndef FEM2D_EMULATE
#include <stdlib.h>

#include "common.cuh"
#endif
#include "fem2d_math.cuh"

namespace gad {
#ifdef FEM2D_EMULATE          // oracle/fem2d_emu.cpp: the kernels on CPU threads; they must be visible to that file
inline namespace emu {
#else
namespace {
#endif

using namespace fem2d;

constexpr int FEM2D_THREADS = 512;
// An evaluation point on a vertex lies in every cell of the vertex's star, so the point pass must keep D hits: the
// launch check bounds D by MAX_HITS.  f2_load<1> packs 2 bits per star cell into one 32-bit mask: D <= 16.
constexpr int MAX_HITS = 16;
static_assert(2 * MAX_HITS <= 32, "f2_load<1>: the star-cell mask has 2 bits per cell in 32 bits");
constexpr int MAX_GAUSS = 16;
constexpr int MAX_ROWS_PER_THREAD = 8;     // CG keeps r / x / Ap of its rows in registers: N <= 8 * 512 (template R)
__host__ __device__ inline int f2_rows_per_thread(int N) {
    const int need = (N + FEM2D_THREADS - 1) / FEM2D_THREADS;
    return need <= 1 ? 1 : (need <= 2 ? 2 : (need <= 4 ? 4 : 8));
}

struct F2Args {
    const int* cells;        // [T,3]
    const unsigned char* is_bc;   // [N]
    const int* star_cell;    // [N,D]
    const int* star_loc;     // [N,D]
    const float* coords;     // [B,N,2]
    const double* cen;       // [B,G,2]
    const double* sc;        // [B,G,2]
    const float* ex;         // [Q]
    const float* ey;         // [Q]
    const float* g_sol;      // [B,Q]   (backward)
    float* coeffs;           // [B,N]
    float* sol;              // [B,Q]
    double* u64;             // [B,N]   forward -> backward
    float* grad;             // [B,N,2] (backward)
    int* cg_iters;           // [B] or null
    int T, N, D, G, K, Q;
};

// A point that passes the (rounded) edge tests of a cell can lie outside the cell's exact bounding box only by the
// rounding error of those tests (~1e-7 / edge length); the margin is orders of magnitude above that, so the prefilter
// never changes which cells count.
constexpr float BOX_MARGIN = 1e-3f;

// Everything the hat function of node m needs from ONE cell of its star, worked out once per node instead of once
// per cubature point (c = m's vertex in the cell, a / b the other two, as phi_star orders them): the three edge
// tests  e?x * P.x + e?y * P.y  against  r?  (inside_count), and the barycentric coordinates of c, a, b at P
// (bary): numerator coefficients = the edge coefficients, base point, denominator; (gx, gy) = grad l_c.
// Same operands, same operations as inside_count / bary: bit-identical decisions and values.
struct StarRec {
    float e1x, e1y, r1, e2x, e2y, r2, e3x, e3y, r3, valid;
    float denc, cx, cy, dena, ax, ay, denb, bx, by, gx, gy;
    float pad[3];
    int ia, ib, ic;
    int pad2;
};
__device__ inline StarRec f2_star_rec(P2 a, P2 b, P2 c, int ia, int ib, int ic) {
    StarRec r;
    r.e1x = a.y - b.y, r.e1y = b.x - a.x;
    r.r1 = FEM_ADD(FEM_MUL(r.e1x, a.x), FEM_MUL(r.e1y, a.y));
    r.e2x = b.y - c.y, r.e2y = c.x - b.x;
    r.r2 = FEM_ADD(FEM_MUL(r.e2x, b.x), FEM_MUL(r.e2y, b.y));
    r.e3x = c.y - a.y, r.e3y = a.x - c.x;
    r.r3 = FEM_ADD(FEM_MUL(r.e3x, c.x), FEM_MUL(r.e3y, c.y));
    r.valid = 1.f;
    r.denc = FEM_ADD(FEM_MUL(r.e1x, c.x - a.x), FEM_MUL(c.y - a.y, r.e1y));
    r.dena = FEM_ADD(FEM_MUL(r.e2x, a.x - b.x), FEM_MUL(a.y - b.y, r.e2y));
    r.denb = FEM_ADD(FEM_MUL(r.e3x, b.x - c.x), FEM_MUL(b.y - c.y, r.e3y));
    r.cx = c.x, r.cy = c.y, r.ax = a.x, r.ay = a.y, r.bx = b.x, r.by = b.y;
    r.gx = r.e1x / r.denc, r.gy = r.e1y / r.denc;
    r.ia = ia, r.ib = ib, r.ic = ic;
    r.pad[0] = r.pad[1] = r.pad[2] = 0.f;
    r.pad2 = 0;
    return r;
}
__device__ inline int f2_rec_inside(const StarRec& r, P2 P) {
    const float l1 = FEM_ADD(FEM_MUL(r.e1x, P.x), FEM_MUL(r.e1y, P.y));
    const float l2 = FEM_ADD(FEM_MUL(r.e2x, P.x), FEM_MUL(r.e2y, P.y));
    const float l3 = FEM_ADD(FEM_MUL(r.e3x, P.x), FEM_MUL(r.e3y, P.y));
    const int left = (l1 >= r.r1) && (l2 >= r.r2) && (l3 >= r.r3);
    const int right = (l1 <= r.r1) && (l2 <= r.r2) && (l3 <= r.r3);
    return left + right;
}
__device__ inline float f2_rec_lc(const StarRec& r, P2 P) {
    return FEM_ADD(1.f, FEM_ADD(FEM_MUL(P.x - r.cx, r.e1x), FEM_MUL(P.y - r.cy, r.e1y)) / r.denc);
}
__device__ inline float f2_rec_la(const StarRec& r, P2 P) {
    return FEM_ADD(1.f, FEM_ADD(FEM_MUL(P.x - r.ax, r.e2x), FEM_MUL(P.y - r.ay, r.e2y)) / r.dena);
}
__device__ inline float f2_rec_lb(const StarRec& r, P2 P) {
    return FEM_ADD(1.f, FEM_ADD(FEM_MUL(P.x - r.bx, r.e3x), FEM_MUL(P.y - r.by, r.e3y)) / r.denb);
}

// Shared memory of one mesh.  `uni` is time-shared: the matrix rows during a CG solve, the bin table during a point pass.
struct F2Smem {
    float* xy;              // [2N]
    unsigned short* cell;   // [T,4]   vertices of every cell (4th entry unused): one 8-byte load
    double* u;              // [N]
    double* b;              // [N]
    double* r;              // [N]     backward: lambda
    double* p;              // [N]
    double* acc;            // [2N]    gradient / g_u accumulators; CG result
    double* red;            // [2][32] partial sums of the block reductions (double-buffered: one barrier each)
    float* bbox;            // [4]     bounding box of the mesh
    GaussPre* gp;           // [MAX_GAUSS] per-Gaussian constants of the forcing
    StarRec* star;          // [warps, D]  star records of the node each warp is working on (load vector phases)
    unsigned char* uni;
    // rows view (RW = D + 2 entries per node, column-major)
    double* coef;           // [RW, N]
    unsigned short* col;    // [RW, N]
    // bin view
    int* bin_ptr;           // [NB + 1]
    int* bin_fill;          // [NB]
    unsigned short* bin_cell;   // [cap]
    int RW, NBX, cap;
};

__host__ __device__ inline size_t f2_align(size_t x) { return (x + 15) & ~(size_t)15; }
__host__ __device__ inline int f2_nbx(int T) {
    int n = 4;
    while (n < 64 && 2 * n * n < T) n *= 2;     // about one or two cells per bin
    return n;
}
__host__ __device__ inline int f2_row_width(int D) { return (D + 2 + 3) & ~3; }   // padded: the CG row loop is unrolled by 4
__host__ __device__ inline size_t f2_rows_bytes(int N, int D) {
    return f2_align((size_t)f2_row_width(D) * N * 8) + f2_align((size_t)f2_row_width(D) * N * 2);
}
__host__ __device__ inline size_t f2_bins_min_bytes(int T) {
    const int nb = f2_nbx(T) * f2_nbx(T);
    return f2_align((size_t)(nb + 1) * 4) + f2_align((size_t)nb * 4) + f2_align((size_t)9 * T * 2);
}
__host__ __device__ inline size_t f2_uni_bytes(int N, int T, int D) {
    const size_t r = f2_rows_bytes(N, D), q = f2_bins_min_bytes(T);
    return r > q ? r : q;
}
__host__ __device__ inline size_t f2_smem_bytes(int N, int T, int D) {
    return f2_align(2 * (size_t)N * 4) + f2_align((size_t)T * 8) + 4 * f2_align((size_t)N * 8) + f2_align(2 * (size_t)N * 8) +
           f2_align(64 * 8) + f2_align(16) + f2_align(MAX_GAUSS * sizeof(GaussPre)) +
           f2_align((size_t)(FEM2D_THREADS / 32) * D * sizeof(StarRec)) + f2_uni_bytes(N, T, D);
}

__device__ inline F2Smem f2_carve(unsigned char* base, int N, int T, int D) {
    F2Smem s;
    size_t o = 0;
    s.xy = reinterpret_cast<float*>(base + o), o += f2_align(2 * (size_t)N * 4);
    s.cell = reinterpret_cast<unsigned short*>(base + o), o += f2_align((size_t)T * 8);
    s.u = reinterpret_cast<double*>(base + o), o += f2_align((size_t)N * 8);
    s.b = reinterpret_cast<double*>(base + o), o += f2_align((size_t)N * 8);
    s.r = reinterpret_cast<double*>(base + o), o += f2_align((size_t)N * 8);
    s.p = reinterpret_cast<double*>(base + o), o += f2_align((size_t)N * 8);
    s.acc = reinterpret_cast<double*>(base + o), o += f2_align(2 * (size_t)N * 8);
    s.red = reinterpret_cast<double*>(base + o), o += f2_align(64 * 8);
    s.bbox = reinterpret_cast<float*>(base + o), o += f2_align(16);
    s.gp = reinterpret_cast<GaussPre*>(base + o), o += f2_align(MAX_GAUSS * sizeof(GaussPre));
    s.star = reinterpret_cast<StarRec*>(base + o), o += f2_align((size_t)(FEM2D_THREADS / 32) * D * sizeof(StarRec));
    s.uni = base + o;
    s.RW = f2_row_width(D);
    s.coef = reinterpret_cast<double*>(s.uni);
    s.col = reinterpret_cast<unsigned short*>(s.uni + f2_align((size_t)s.RW * N * 8));
    s.NBX = f2_nbx(T);
    const int nb = s.NBX * s.NBX;
    s.bin_ptr = reinterpret_cast<int*>(s.uni);
    s.bin_fill = reinterpret_cast<int*>(s.uni + f2_align((size_t)(nb + 1) * 4));
    const size_t head = f2_align((size_t)(nb + 1) * 4) + f2_align((size_t)nb * 4);
    s.bin_cell = reinterpret_cast<unsigned short*>(s.uni + head);
    s.cap = (int)((f2_uni_bytes(N, T, D) - head) / 2);
    return s;
}

__device__ inline P2 f2_pt(const float* xy, int i) { return P2{xy[2 * i], xy[2 * i + 1]}; }

// Optional phase timeline of CTA 0 (profiling aid, GAD_FEM2D_TRACE=1: f2_launch prints it to stderr)
#ifndef FEM2D_EMULATE
__device__ long long g_f2_trace[2][16];
__device__ int g_f2_trace_on;
__device__ __forceinline__ void f2_mark(int kernel, int slot) {
    if (g_f2_trace_on && blockIdx.x == 0 && threadIdx.x == 0) {
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_f2_trace[kernel][slot] = t;
    }
}
#else
inline void f2_mark(int, int) {}
#endif

// fixed-order block sum (every thread gets the result); `which` alternates between two buffers so that consecutive
// reductions need one barrier each
__device__ double f2_block_sum(double v, double* red, int which) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    double* buf = red + 32 * (which & 1);
    if ((threadIdx.x & 31) == 0) buf[w] = v;
    __syncthreads();
    double s = 0.0;
    for (int k = 0; k < nw; ++k) s += buf[k];
    return s;
}

__device__ void f2_geometry(const F2Args& a, const F2Smem& s, int mesh) {
    const float* c = a.coords + (size_t)mesh * a.N * 2;
    for (int i = threadIdx.x; i < 2 * a.N; i += blockDim.x) s.xy[i] = c[i];
    for (int t = threadIdx.x; t < a.T; t += blockDim.x) {
        s.cell[4 * t] = (unsigned short)a.cells[3 * t];
        s.cell[4 * t + 1] = (unsigned short)a.cells[3 * t + 1];
        s.cell[4 * t + 2] = (unsigned short)a.cells[3 * t + 2];
        s.cell[4 * t + 3] = 0;
    }
    __syncthreads();
}

__device__ inline Tri f2_tri(const F2Smem& s, int t) {
    return tri_geometry(f2_pt(s.xy, s.cell[4 * t]), f2_pt(s.xy, s.cell[4 * t + 1]), f2_pt(s.xy, s.cell[4 * t + 2]));
}

// Interior stiffness matrix K_II as padded rows in shared memory: row i holds, for every interior neighbour j
// (i itself included), K_ij = sum over the cells of the star of i that contain j of the fp32 local entry, added in
// fp64 in ascending star order.  Unused slots: column i, coefficient 0.  Dirichlet rows are empty.
__device__ void f2_build_rows(const F2Args& a, const F2Smem& s) {
    const int N = a.N, RW = s.RW;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        for (int q = 0; q < RW; ++q) {
            s.coef[(size_t)q * N + i] = 0.0;
            s.col[(size_t)q * N + i] = (unsigned short)i;
        }
        if (a.is_bc[i]) continue;
        int used = 0;
        for (int d = 0; d < a.D; ++d) {
            const int t = a.star_cell[i * a.D + d];
            if (t < 0) continue;
            const int k = a.star_loc[i * a.D + d];
            const Tri g = f2_tri(s, t);
            for (int kk = 0; kk < 3; ++kk) {
                const int j = s.cell[4 * t + kk];
                if (a.is_bc[j]) continue;
                int q = 0;
                while (q < used && s.col[(size_t)q * N + i] != j) ++q;
                if (q == used) {
                    if (used == RW) continue;      // cannot happen: a star of D cells has at most D + 2 vertices
                    s.col[(size_t)q * N + i] = (unsigned short)j;
                    ++used;
                }
                s.coef[(size_t)q * N + i] += (double)tri_k(g, k, kk);
            }
        }
    }
    __syncthreads();
}

// conjugate gradients on K_II x = b (b in s.b, zero on Dirichlet nodes; rows built by f2_build_rows); x -> out
// (all threads see it after return).  Thread t owns rows t, t + blockDim, ...: r, x and Ap of those rows never
// leave its registers; only the search direction p is exchanged through shared memory.
template <int R>
__device__ int f2_cg(const F2Args& a, const F2Smem& s, double* out) {
    const int N = a.N, RW = s.RW, nthr = blockDim.x;
    double r[R], x[R], Ap[R];
    double l = 0.0;
#pragma unroll
    for (int m = 0; m < R; ++m) {
        const int i = threadIdx.x + m * nthr;
        x[m] = 0.0;
        r[m] = (i < N) ? s.b[i] : 0.0;
        if (i < N) s.p[i] = r[m];
        l += r[m] * r[m];
    }
    int which = 0;
    double rr = f2_block_sum(l, s.red, which++);      // its barrier also publishes p
    const double bb = rr;
    int it = 0;
    for (; it < 20 * N && rr > 1e-28 * bb && rr > 0.0; ++it) {
        l = 0.0;
#pragma unroll
        for (int m = 0; m < R; ++m) {
            const int i = threadIdx.x + m * nthr;
            double acc = 0.0;
            if (i < N) {
                for (int q = 0; q < RW; q += 4) {          // all loads of four entries in flight before the first FMA
                    const unsigned short* cq = s.col + (size_t)q * N + i;
                    const double* kq = s.coef + (size_t)q * N + i;
                    const int c0 = cq[0], c1 = cq[N], c2 = cq[2 * N], c3 = cq[3 * N];
                    const double k0 = kq[0], k1 = kq[N], k2 = kq[2 * N], k3 = kq[3 * N];
                    const double p0 = s.p[c0], p1 = s.p[c1], p2 = s.p[c2], p3 = s.p[c3];
                    acc += k0 * p0;
                    acc += k1 * p1;
                    acc += k2 * p2;
                    acc += k3 * p3;
                }
                l += s.p[i] * acc;
            }
            Ap[m] = acc;
        }
        const double alpha = rr / f2_block_sum(l, s.red, which++);
        l = 0.0;
#pragma unroll
        for (int m = 0; m < R; ++m) {
            const int i = threadIdx.x + m * nthr;
            if (i < N) {
                x[m] += alpha * s.p[i];
                r[m] -= alpha * Ap[m];
                l += r[m] * r[m];
            }
        }
        const double rr2 = f2_block_sum(l, s.red, which++);   // after this barrier nobody reads the old p any more
        const double beta = rr2 / rr;
#pragma unroll
        for (int m = 0; m < R; ++m) {
            const int i = threadIdx.x + m * nthr;
            if (i < N) s.p[i] = r[m] + beta * s.p[i];
        }
        rr = rr2;
        __syncthreads();
    }
#pragma unroll
    for (int m = 0; m < R; ++m) {
        const int i = threadIdx.x + m * nthr;
        if (i < N) out[i] = x[m];
    }
    __syncthreads();
    return it;
}

__device__ void f2_star_box(const F2Args& a, const F2Smem& s, int i, float& lx, float& ly, float& hx, float& hy) {
    lx = ly = INFINITY;
    hx = hy = -INFINITY;
    for (int d = 0; d < a.D; ++d) {
        const int t = a.star_cell[i * a.D + d];
        if (t < 0) continue;
        for (int kk = 0; kk < 3; ++kk) {
            const P2 p = f2_pt(s.xy, s.cell[4 * t + kk]);
            lx = fminf(lx, p.x), ly = fminf(ly, p.y), hx = fmaxf(hx, p.x), hy = fmaxf(hy, p.y);
        }
    }
}

// grad[v] += -coef * l_v(P) * g_c for the three vertices of cell t (c = local vertex k)
__device__ void f2_scatter(const F2Args& a, const F2Smem& s, int t, int k, P2 P, double coef) {
    const int ic = s.cell[4 * t + k], ia = s.cell[4 * t + (k + 2) % 3], ib = s.cell[4 * t + (k + 1) % 3];
    const P2 pa = f2_pt(s.xy, ia), pb = f2_pt(s.xy, ib), pc = f2_pt(s.xy, ic);
    float gx, gy, tx, ty;
    const float lc = bary(P, pa, pb, pc, &gx, &gy);
    const float la = bary(P, pb, pc, pa, &tx, &ty);
    const float lb = bary(P, pc, pa, pb, &tx, &ty);
    atomicAdd(&s.acc[2 * ia], -coef * (double)la * (double)gx);
    atomicAdd(&s.acc[2 * ia + 1], -coef * (double)la * (double)gy);
    atomicAdd(&s.acc[2 * ib], -coef * (double)lb * (double)gx);
    atomicAdd(&s.acc[2 * ib + 1], -coef * (double)lb * (double)gy);
    atomicAdd(&s.acc[2 * ic], -coef * (double)lc * (double)gx);
    atomicAdd(&s.acc[2 * ic + 1], -coef * (double)lc * (double)gy);
}

// inflated bounding box of a cell (the prefilter of the point location, see BOX_MARGIN)
__device__ inline void f2_cell_box(const F2Smem& s, int t, float& lx, float& ly, float& hx, float& hy) {
    const P2 p0 = f2_pt(s.xy, s.cell[4 * t]), p1 = f2_pt(s.xy, s.cell[4 * t + 1]), p2 = f2_pt(s.xy, s.cell[4 * t + 2]);
    lx = fminf(p0.x, fminf(p1.x, p2.x)) - BOX_MARGIN, ly = fminf(p0.y, fminf(p1.y, p2.y)) - BOX_MARGIN;
    hx = fmaxf(p0.x, fmaxf(p1.x, p2.x)) + BOX_MARGIN, hy = fmaxf(p0.y, fmaxf(p1.y, p2.y)) + BOX_MARGIN;
}
// bin coordinate of x: monotone in x, so lo <= x <= hi implies bin(lo) <= bin(x) <= bin(hi)
__device__ inline int f2_bin(float x, float lo, float inv, int nbx) {
    const float f = floorf((x - lo) * inv);
    return f < 0.f ? 0 : (f > (float)(nbx - 1) ? nbx - 1 : (int)f);
}

// Uniform bin table over the mesh's bounding box: every cell is listed in the bins its inflated bounding box
// overlaps (count, exclusive scan, fill).  Returns false (all threads) when the table does not fit the shared
// memory left for it; the point pass then scans all cells.
__device__ bool f2_build_bins(const F2Args& a, const F2Smem& s) {
    const int nbx = s.NBX, nb = nbx * nbx;
    if (threadIdx.x < 32) {
        float lx = INFINITY, ly = INFINITY, hx = -INFINITY, hy = -INFINITY;
        for (int i = threadIdx.x; i < a.N; i += 32) {
            lx = fminf(lx, s.xy[2 * i]), hx = fmaxf(hx, s.xy[2 * i]);
            ly = fminf(ly, s.xy[2 * i + 1]), hy = fmaxf(hy, s.xy[2 * i + 1]);
        }
        for (int d = 16; d > 0; d >>= 1) {
            lx = fminf(lx, (float)__shfl_xor_sync(0xffffffffu, (double)lx, d));
            ly = fminf(ly, (float)__shfl_xor_sync(0xffffffffu, (double)ly, d));
            hx = fmaxf(hx, (float)__shfl_xor_sync(0xffffffffu, (double)hx, d));
            hy = fmaxf(hy, (float)__shfl_xor_sync(0xffffffffu, (double)hy, d));
        }
        if (threadIdx.x == 0) s.bbox[0] = lx, s.bbox[1] = ly, s.bbox[2] = hx, s.bbox[3] = hy;
    }
    for (int k = threadIdx.x; k < nb; k += blockDim.x) s.bin_fill[k] = 0;
    __syncthreads();
    const float LX = s.bbox[0], LY = s.bbox[1];
    const float ivx = (float)nbx / fmaxf(s.bbox[2] - LX, 1e-30f), ivy = (float)nbx / fmaxf(s.bbox[3] - LY, 1e-30f);
    for (int t = threadIdx.x; t < a.T; t += blockDim.x) {
        float lx, ly, hx, hy;
        f2_cell_box(s, t, lx, ly, hx, hy);
        const int x0 = f2_bin(lx, LX, ivx, nbx), x1 = f2_bin(hx, LX, ivx, nbx);
        const int y0 = f2_bin(ly, LY, ivy, nbx), y1 = f2_bin(hy, LY, ivy, nbx);
        for (int by = y0; by <= y1; ++by)
            for (int bx = x0; bx <= x1; ++bx) atomicAdd(&s.bin_fill[by * nbx + bx], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int k = 0; k < nb; ++k) {
            s.bin_ptr[k] = run;
            run += s.bin_fill[k];
        }
        s.bin_ptr[nb] = run;
    }
    __syncthreads();
    const bool fits = s.bin_ptr[nb] <= s.cap;
    for (int k = threadIdx.x; k < nb; k += blockDim.x) s.bin_fill[k] = s.bin_ptr[k];
    __syncthreads();
    if (fits)
        for (int t = threadIdx.x; t < a.T; t += blockDim.x) {
            float lx, ly, hx, hy;
            f2_cell_box(s, t, lx, ly, hx, hy);
            const int x0 = f2_bin(lx, LX, ivx, nbx), x1 = f2_bin(hx, LX, ivx, nbx);
            const int y0 = f2_bin(ly, LY, ivy, nbx), y1 = f2_bin(hy, LY, ivy, nbx);
            for (int by = y0; by <= y1; ++by)
                for (int bx = x0; bx <= x1; ++bx) s.bin_cell[atomicAdd(&s.bin_fill[by * nbx + bx], 1)] = (unsigned short)t;
        }
    __syncthreads();
    return fits;
}

__device__ inline void f2_try_cell(const F2Smem& s, P2 P, int t, int* ht, int* hm, int& nh) {
    float lx, ly, hx, hy;
    f2_cell_box(s, t, lx, ly, hx, hy);
    if (P.x < lx || P.x > hx || P.y < ly || P.y > hy) return;
    const int mult = inside_count(P, f2_pt(s.xy, s.cell[4 * t + 2]), f2_pt(s.xy, s.cell[4 * t + 1]), f2_pt(s.xy, s.cell[4 * t]));
    if (mult && nh < MAX_HITS) ht[nh] = t, hm[nh] = mult, ++nh;
}

// The evaluation points of this thread: hit cells (in ascending cell order, as the reference's scan finds them), per
// distinct vertex value / repeat (phim, difFEM_2d.py:28-60).
// MODE 0: sol[q].  MODE 1: g_u accumulation (s.acc[v]).  MODE 2: interpolation term of the gradient (s.acc[2v..]).
template <int MODE>
__device__ void f2_points(const F2Args& a, const F2Smem& s, int mesh, bool bins) {
    const int nbx = s.NBX;
    const float LX = s.bbox[0], LY = s.bbox[1];
    const float ivx = (float)nbx / fmaxf(s.bbox[2] - LX, 1e-30f), ivy = (float)nbx / fmaxf(s.bbox[3] - LY, 1e-30f);
    for (int q = threadIdx.x; q < a.Q; q += blockDim.x) {
        const P2 P{a.ex[q], a.ey[q]};
        int ht[MAX_HITS], hm[MAX_HITS], nh = 0;
        if (bins) {
            const int k = f2_bin(P.y, LY, ivy, nbx) * nbx + f2_bin(P.x, LX, ivx, nbx);
            for (int e = s.bin_ptr[k]; e < s.bin_ptr[k + 1]; ++e) f2_try_cell(s, P, s.bin_cell[e], ht, hm, nh);
            for (int x = 1; x < nh; ++x) {                     // the bin lists are unordered: sort the hits by cell id
                const int t = ht[x], m = hm[x];
                int y = x - 1;
                for (; y >= 0 && ht[y] > t; --y) ht[y + 1] = ht[y], hm[y + 1] = hm[y];
                ht[y + 1] = t, hm[y + 1] = m;
            }
        } else {
            for (int t = 0; t < a.T && nh < MAX_HITS; ++t) f2_try_cell(s, P, t, ht, hm, nh);
        }
        const double gq = (MODE == 0) ? 0.0 : (double)a.g_sol[(size_t)mesh * a.Q + q];
        double val = 0.0;
        for (int h = 0; h < nh; ++h)
            for (int k = 0; k < 3; ++k) {
                const int v = s.cell[4 * ht[h] + k];
                bool first = true;
                for (int h2 = 0; h2 < h && first; ++h2)
                    for (int k2 = 0; k2 < 3; ++k2)
                        if (s.cell[4 * ht[h2] + k2] == v) first = false;
                if (!first) continue;
                float num = 0.f, rep = 0.f;
                for (int h2 = h; h2 < nh; ++h2)
                    for (int k2 = 0; k2 < 3; ++k2) {
                        const int t2 = ht[h2];
                        if (s.cell[4 * t2 + k2] != v) continue;
                        float gx, gy;
                        const float inc = (float)hm[h2] * bary(P, f2_pt(s.xy, s.cell[4 * t2 + (k2 + 2) % 3]),
                                                               f2_pt(s.xy, s.cell[4 * t2 + (k2 + 1) % 3]), f2_pt(s.xy, v), &gx, &gy);
                        num += inc;
                        rep += (inc > 0.f) ? 1.f : 0.f;
                    }
                if (rep == 0.f) rep = 1.f;
                const float phi = num / rep;
                const double uv = (double)(float)s.u[v];
                if (MODE == 0) val += uv * (double)phi;
                if (MODE == 1) atomicAdd(&s.acc[v], gq * (double)phi);
                if (MODE == 2)
                    for (int h2 = h; h2 < nh; ++h2)
                        for (int k2 = 0; k2 < 3; ++k2)
                            if (s.cell[4 * ht[h2] + k2] == v) f2_scatter(a, s, ht[h2], k2, P, uv * gq * hm[h2] / (double)rep);
            }
        if (MODE == 0) a.sol[(size_t)mesh * a.Q + q] = (float)val;
    }
    __syncthreads();
}

// load vector (MODE 0: rhs into s.b as doubles) or its gradient term (MODE 1: needs lambda in s.r)
template <int MODE>
__device__ void f2_load(const F2Args& a, const F2Smem& s, const double* cen, const double* sc) {
    const int n = simpson_n(a.K);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if (threadIdx.x < a.G) s.gp[threadIdx.x] = gauss_pre(cen, sc, threadIdx.x);
    __syncthreads();
    for (int i = warp; i < a.N; i += nw) {
        if (a.is_bc[i]) {
            if (MODE == 0 && lane == 0) s.b[i] = u_true((double)s.xy[2 * i], (double)s.xy[2 * i + 1], cen, sc, a.G);
            continue;
        }
        // star records of node i: lane d builds the record of star cell d (and the bounding box comes with them)
        StarRec* rec = s.star + (size_t)warp * a.D;
        __syncwarp();                      // the previous node's records are no longer read
        if (lane < a.D) {
            const int t = a.star_cell[i * a.D + lane];
            if (t < 0) {
                rec[lane].valid = 0.f;
            } else {
                const int k = a.star_loc[i * a.D + lane];
                const int ic = s.cell[4 * t + k], ia = s.cell[4 * t + (k + 2) % 3], ib = s.cell[4 * t + (k + 1) % 3];
                rec[lane] = f2_star_rec(f2_pt(s.xy, ia), f2_pt(s.xy, ib), f2_pt(s.xy, ic), ia, ib, ic);
            }
        }
        __syncwarp();
        float lx = INFINITY, ly = INFINITY, hx = -INFINITY, hy = -INFINITY;
        for (int d = 0; d < a.D; ++d) {
            if (rec[d].valid == 0.f) continue;
            lx = fminf(lx, fminf(rec[d].ax, fminf(rec[d].bx, rec[d].cx))), hx = fmaxf(hx, fmaxf(rec[d].ax, fmaxf(rec[d].bx, rec[d].cx)));
            ly = fminf(ly, fminf(rec[d].ay, fminf(rec[d].by, rec[d].cy))), hy = fmaxf(hy, fmaxf(rec[d].ay, fmaxf(rec[d].by, rec[d].cy)));
        }
        const double hh = (double)((hx - lx) / (float)(n - 1)) * (double)((hy - ly) / (float)(n - 1)) / 9.0;
        if (MODE == 0) {
            double part = 0.0;
            for (int pq = lane; pq < n * n; pq += 32) {
                const int ia = pq / n, ib = pq % n;
                const P2 P{linspace_at(lx, hx, n, ia), linspace_at(ly, hy, n, ib)};
                float out = 0.f, rep = 0.f;           // phi_star (fem2d_math.cuh) over the records
                for (int d = 0; d < a.D; ++d) {
                    if (rec[d].valid == 0.f) continue;
                    const int mult = f2_rec_inside(rec[d], P);
                    if (!mult) continue;
                    const float inc = (float)mult * f2_rec_lc(rec[d], P);
                    out += inc;
                    rep += (inc > 0.f) ? 1.f : 0.f;
                }
                if (rep == 0.f) rep = 1.f;
                const float phi = out / rep;
                const float f = (float)forcing_pre((double)P.x, (double)P.y, s.gp, sc, a.G);
                const double w = (double)(simpson_w(n, ia) * simpson_w(n, ib));
                part += (double)(phi * f) * w;
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) part += __shfl_xor_sync(0xffffffffu, part, d);
            if (lane == 0) s.b[i] = (double)(float)(part * hh);
        } else {
            // gradient term: every lane's points contribute to the SAME few vertices (those of the star of i), so the
            // contributions are summed over the warp per star cell first (registers + shuffles) and only lane 0
            // touches the fp64 accumulators in shared memory (a compare-and-swap loop per add)
            constexpr int PTS = 3;
            for (int base = 0; base < n * n; base += 32 * PTS) {
                P2 Pm[PTS];
                double cm[PTS];
                unsigned mm[PTS];
#pragma unroll
                for (int m = 0; m < PTS; ++m) {
                    const int pq = base + m * 32 + lane;
                    cm[m] = 0.0;
                    mm[m] = 0;
                    Pm[m] = P2{0.f, 0.f};
                    if (pq < n * n) {
                        const int ia = pq / n, ib = pq % n;
                        Pm[m] = P2{linspace_at(lx, hx, n, ia), linspace_at(ly, hy, n, ib)};
                        // phi_star's repeat count, keeping which star cells contain the point (2 bits per cell)
                        float rep = 0.f;
                        unsigned mask = 0;
                        for (int d = 0; d < a.D; ++d) {
                            if (rec[d].valid == 0.f) continue;
                            const int mult = f2_rec_inside(rec[d], Pm[m]);
                            if (!mult) continue;
                            mask |= (unsigned)mult << (2 * d);
                            const float inc = (float)mult * f2_rec_lc(rec[d], Pm[m]);
                            rep += (inc > 0.f) ? 1.f : 0.f;
                        }
                        if (rep == 0.f) rep = 1.f;
                        mm[m] = mask;
                        const float f = (float)forcing_pre((double)Pm[m].x, (double)Pm[m].y, s.gp, sc, a.G);
                        const double w = (double)(simpson_w(n, ia) * simpson_w(n, ib));
                        cm[m] = s.r[i] * hh * w * (double)f / (double)rep;
                    }
                }
                for (int d = 0; d < a.D; ++d) {
                    if (rec[d].valid == 0.f) continue;
                    const float gx = rec[d].gx, gy = rec[d].gy;
                    double g[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
                    for (int m = 0; m < PTS; ++m) {
                        const int mult = (int)((mm[m] >> (2 * d)) & 3u);
                        if (!mult || cm[m] == 0.0) continue;
                        const double coef = cm[m] * mult;
                        const float lc = f2_rec_lc(rec[d], Pm[m]);
                        const float la = f2_rec_la(rec[d], Pm[m]);
                        const float lb = f2_rec_lb(rec[d], Pm[m]);
                        g[0] += -coef * (double)la * (double)gx, g[1] += -coef * (double)la * (double)gy;
                        g[2] += -coef * (double)lb * (double)gx, g[3] += -coef * (double)lb * (double)gy;
                        g[4] += -coef * (double)lc * (double)gx, g[5] += -coef * (double)lc * (double)gy;
                    }
#pragma unroll
                    for (int c = 0; c < 6; ++c)
#pragma unroll
                        for (int sh = 16; sh > 0; sh >>= 1) g[c] += __shfl_xor_sync(0xffffffffu, g[c], sh);
                    if (lane < 6) {          // after the butterfly every lane holds the sums: one add per lane, in parallel
                        const int v = lane < 2 ? rec[d].ia : (lane < 4 ? rec[d].ib : rec[d].ic);
                        const double gv = lane == 0 ? g[0] : (lane == 1 ? g[1] : (lane == 2 ? g[2] : (lane == 3 ? g[3] : (lane == 4 ? g[4] : g[5]))));
                        atomicAdd(&s.acc[2 * v + (lane & 1)], gv);
                    }
                }
            }
        }
    }
    __syncthreads();
}

// right-hand side of the interior system from rhs (s.b) and the Dirichlet values: b_i = -rhs_i - sum_B K_ij u_j
__device__ void f2_interior_rhs(const F2Args& a, const F2Smem& s) {
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) s.u[i] = a.is_bc[i] ? s.b[i] : 0.0;
    __syncthreads();
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) {
        double v = 0.0;
        if (!a.is_bc[i]) {
            v = -s.b[i];
            for (int d = 0; d < a.D; ++d) {
                const int t = a.star_cell[i * a.D + d];
                if (t < 0) continue;
                const int k = a.star_loc[i * a.D + d];
                const Tri g = f2_tri(s, t);
                for (int kk = 0; kk < 3; ++kk) {
                    const int j = s.cell[4 * t + kk];
                    if (a.is_bc[j]) v -= (double)tri_k(g, k, kk) * s.u[j];
                }
            }
        }
        s.p[i] = v;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) s.b[i] = s.p[i];
    __syncthreads();
}

template <int R>
__global__ void __launch_bounds__(FEM2D_THREADS) k_fem2d_fwd(F2Args a) {
    extern __shared__ __align__(16) unsigned char f2_raw[];
    const F2Smem s = f2_carve(f2_raw, a.N, a.T, a.D);
    const int mesh = blockIdx.x;
    const double* cen = a.cen + (size_t)mesh * a.G * 2;
    const double* sc = a.sc + (size_t)mesh * a.G * 2;
    f2_mark(0, 0);
    f2_geometry(a, s, mesh);
    f2_mark(0, 1);
    f2_load<0>(a, s, cen, sc);
    f2_mark(0, 2);
    f2_interior_rhs(a, s);
    f2_build_rows(a, s);
    f2_mark(0, 3);
    const int it = f2_cg<R>(a, s, s.acc);              // interior solution in s.acc[0..N)
    f2_mark(0, 4);
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) {
        if (!a.is_bc[i]) s.u[i] = s.acc[i];
        a.coeffs[(size_t)mesh * a.N + i] = (float)s.u[i];
        a.u64[(size_t)mesh * a.N + i] = s.u[i];
    }
    __syncthreads();
    const bool bins = f2_build_bins(a, s);           // the rows are no longer needed: their memory holds the bins
    f2_mark(0, 5);
    f2_points<0>(a, s, mesh, bins);
    f2_mark(0, 6);
    if (a.cg_iters && threadIdx.x == 0) a.cg_iters[mesh] = it;
}

template <int R>
__global__ void __launch_bounds__(FEM2D_THREADS) k_fem2d_bwd(F2Args a) {
    extern __shared__ __align__(16) unsigned char f2_raw[];
    const F2Smem s = f2_carve(f2_raw, a.N, a.T, a.D);
    const int mesh = blockIdx.x;
    const double* cen = a.cen + (size_t)mesh * a.G * 2;
    const double* sc = a.sc + (size_t)mesh * a.G * 2;
    f2_geometry(a, s, mesh);
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) s.u[i] = a.u64[(size_t)mesh * a.N + i];
    for (int i = threadIdx.x; i < 2 * a.N; i += blockDim.x) s.acc[i] = 0.0;
    __syncthreads();
    f2_mark(1, 0);
    bool bins = f2_build_bins(a, s);
    f2_mark(1, 1);
    f2_points<1>(a, s, mesh, bins);                  // g_u in s.acc[0..N)
    f2_mark(1, 2);
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) s.b[i] = a.is_bc[i] ? 0.0 : -s.acc[i];
    __syncthreads();
    f2_build_rows(a, s);                             // (overwrites the bins)
    f2_mark(1, 3);
    double* lam = s.acc + a.N;                       // second half of the accumulator array, free until the scatter
    f2_cg<R>(a, s, lam);                             // K_II lambda_I = -g_I
    f2_mark(1, 4);
    // keep lambda in s.r (zero on Dirichlet nodes), then reuse s.acc as the gradient accumulator
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) s.b[i] = a.is_bc[i] ? 0.0 : lam[i];
    __syncthreads();
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) s.r[i] = s.b[i];
    for (int i = threadIdx.x; i < 2 * a.N; i += blockDim.x) s.acc[i] = 0.0;
    __syncthreads();
    bins = f2_build_bins(a, s);
    f2_mark(1, 5);
    f2_points<2>(a, s, mesh, bins);                  // interpolation term
    f2_mark(1, 6);
    f2_load<1>(a, s, cen, sc);                       // load-vector term
    f2_mark(1, 7);
    for (int t = threadIdx.x; t < a.T; t += blockDim.x) {      // matrix term
        const Tri g = f2_tri(s, t);
        double Glx = 0, Gly = 0, Gux = 0, Guy = 0;
        for (int k = 0; k < 3; ++k) {
            const int v = s.cell[4 * t + k];
            Glx += s.r[v] * g.gx[k], Gly += s.r[v] * g.gy[k];
            Gux += s.u[v] * g.gx[k], Guy += s.u[v] * g.gy[k];
        }
        const double dot = Glx * Gux + Gly * Guy;
        for (int k = 0; k < 3; ++k) {
            const int v = s.cell[4 * t + k];
            const double gx = g.gx[k], gy = g.gy[k];
            const double gGu = gx * Gux + gy * Guy, gGl = gx * Glx + gy * Gly;
            atomicAdd(&s.acc[2 * v], (double)g.area * (dot * gx - gGu * Glx - gGl * Gux));
            atomicAdd(&s.acc[2 * v + 1], (double)g.area * (dot * gy - gGu * Gly - gGl * Guy));
        }
    }
    __syncthreads();
    f2_mark(1, 8);
    for (int i = threadIdx.x; i < 2 * a.N; i += blockDim.x) a.grad[(size_t)mesh * a.N * 2 + i] = (float)s.acc[i];
}

#ifndef FEM2D_EMULATE
int f2_launch(const F2Args& a, int B, bool backward, cudaStream_t st) {
    const size_t bytes = f2_smem_bytes(a.N, a.T, a.D);
    GAD_CHECK_ARG((int)bytes <= smem_optin_bytes(), "fem2d: a mesh of %d nodes / %d cells needs %zu B of shared memory", a.N, a.T,
                  bytes);
    GAD_CHECK_ARG(a.G <= MAX_GAUSS && a.D <= MAX_HITS, "fem2d: at most %d Gaussians and %d cells per node (got %d, %d)",
                  MAX_GAUSS, MAX_HITS, a.G, a.D);
    GAD_CHECK_ARG(a.N <= MAX_ROWS_PER_THREAD * FEM2D_THREADS && a.N <= 65535 && a.T <= 65535,
                  "fem2d: %d nodes / %d cells exceed the kernel's limits (%d nodes, 16-bit indices)", a.N, a.T,
                  MAX_ROWS_PER_THREAD * FEM2D_THREADS);
    static const int trace = getenv("GAD_FEM2D_TRACE") ? atoi(getenv("GAD_FEM2D_TRACE")) : 0;
    if (trace) {
        GAD_CUDA(cudaMemcpyToSymbolAsync(g_f2_trace_on, &trace, sizeof(int), 0, cudaMemcpyHostToDevice, st));
    }
    const int R = f2_rows_per_thread(a.N);
#define F2_LAUNCH(K_)                                                                                        \
    do {                                                                                                     \
        GAD_CUDA(cudaFuncSetAttribute(K_, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));         \
        K_<<<B, FEM2D_THREADS, bytes, st>>>(a);                                                              \
    } while (0)
    if (backward) {
        if (R == 1) F2_LAUNCH(k_fem2d_bwd<1>);
        else if (R == 2) F2_LAUNCH(k_fem2d_bwd<2>);
        else if (R == 4) F2_LAUNCH(k_fem2d_bwd<4>);
        else F2_LAUNCH(k_fem2d_bwd<8>);
    } else {
        if (R == 1) F2_LAUNCH(k_fem2d_fwd<1>);
        else if (R == 2) F2_LAUNCH(k_fem2d_fwd<2>);
        else if (R == 4) F2_LAUNCH(k_fem2d_fwd<4>);
        else F2_LAUNCH(k_fem2d_fwd<8>);
    }
#undef F2_LAUNCH
    if (trace) {
        long long h[2][16];
        GAD_CUDA(cudaStreamSynchronize(st));
        GAD_CUDA(cudaMemcpyFromSymbol(h, g_f2_trace, sizeof(h)));
        const int k = backward ? 1 : 0, n = backward ? 9 : 7;
        static const char* names[2][9] = {{"geometry", "load", "rhs+rows", "cg", "bins", "points", "", "", ""},
                                          {"bins", "points g_u", "rows", "cg", "bins", "points grad", "load grad", "matrix", ""}};
        fprintf(stderr, "[fem2d %s, CTA 0, us]", backward ? "bwd" : "fwd");
        for (int i = 0; i + 1 < n; ++i) fprintf(stderr, " %s %.1f", names[k][i], (h[k][i + 1] - h[k][i]) * 1e-3);
        fprintf(stderr, "\n");
    }
    GAD_LAUNCH_CHECK();
    return GAD_OK;
}
#endif

}  // namespace
}  // namespace gad

#ifndef FEM2D_EMULATE
using namespace gad;

extern "C" int gad_fem2d_fwd(const int32_t* cells, int32_t T, const uint8_t* is_bc, int32_t N, const int32_t* star_cell,
                             const int32_t* star_loc, int32_t D, const float* coords, const double* centers, const double* scales,
                             int32_t G, int32_t B, int32_t load_quad_points, const float* eval_x, const float* eval_y, int32_t Q,
                             float* coeffs, float* sol, double* u64, int32_t* cg_iters, void* stream) {
    GAD_CHECK_ARG(cells && is_bc && star_cell && star_loc && coords && centers && scales && eval_x && eval_y && coeffs && sol && u64,
                  "gad_fem2d_fwd: null argument");
    GAD_CHECK_ARG(T > 0 && N > 0 && D > 0 && G > 0 && B > 0 && Q > 0 && load_quad_points > 0, "gad_fem2d_fwd: bad sizes");
    F2Args a = {};
    a.cells = cells, a.is_bc = is_bc, a.star_cell = star_cell, a.star_loc = star_loc, a.coords = coords, a.cen = centers, a.sc = scales;
    a.ex = eval_x, a.ey = eval_y, a.coeffs = coeffs, a.sol = sol, a.u64 = u64, a.cg_iters = cg_iters;
    a.T = T, a.N = N, a.D = D, a.G = G, a.K = load_quad_points, a.Q = Q;
    return f2_launch(a, B, false, as_stream(stream));
}

extern "C" int gad_fem2d_bwd(const int32_t* cells, int32_t T, const uint8_t* is_bc, int32_t N, const int32_t* star_cell,
                             const int32_t* star_loc, int32_t D, const float* coords, const double* centers, const double* scales,
                             int32_t G, int32_t B, int32_t load_quad_points, const float* eval_x, const float* eval_y, int32_t Q,
                             const double* u64, const float* g_sol, float* grad, void* stream) {
    GAD_CHECK_ARG(cells && is_bc && star_cell && star_loc && coords && centers && scales && eval_x && eval_y && u64 && g_sol && grad,
                  "gad_fem2d_bwd: null argument");
    GAD_CHECK_ARG(T > 0 && N > 0 && D > 0 && G > 0 && B > 0 && Q > 0 && load_quad_points > 0, "gad_fem2d_bwd: bad sizes");
    F2Args a = {};
    a.cells = cells, a.is_bc = is_bc, a.star_cell = star_cell, a.star_loc = star_loc, a.coords = coords, a.cen = centers, a.sc = scales;
    a.ex = eval_x, a.ey = eval_y, a.g_sol = g_sol, a.u64 = const_cast<double*>(u64), a.grad = grad;
    a.T = T, a.N = N, a.D = D, a.G = G, a.K = load_quad_points, a.Q = Q;
    return f2_launch(a, B, true, as_stream(stream));
}
#endif  // FEM2D_EMULATE
