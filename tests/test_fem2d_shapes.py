"""The 2-D FEM kernels (csrc/fem2d.cu) at the shapes the fixtures of tests/test_fem2d_gpu.py never reach: the
production batch (256 distinct jittered 30x30 meshes, 101-point load cubature, 101x101 evaluation grid), every CG
template a mesh that fits in shared memory can select, graded meshes, the quadrature and Gaussian limits, and
vertices of more than 12 cells.

References, per mesh:
  * forward (coefficients, solution): oracle/fem2d_fast.py in fp64.  The forward is continuous in the mesh points,
    so more precision is a valid reference.
  * gradient with respect to the mesh points: NOT fp64.  It jumps across element edges, and cubature and evaluation
    points lie on edges, so which side a point falls on is decided by fp32 rounding (DESIGN section 11); fp64 and fp32
    gradients of the same formulas differ by 3e-2 relative on a jittered 30x30 mesh.  Two references that make the
    kernels' tie decisions instead: the sequential host harness (oracle/fem2d_host.cpp, the same fem2d_math.cuh
    arithmetic with an fp64 CG) at 1e-5, and autograd through oracle/fem2d_fast.py in fp32 (other code, other
    summation order, an fp32 LU solve) at 2e-4: on the jittered meshes below that reference is itself up to 1.2e-4
    from the host harness, which the kernels match to 5e-6.

The tests without the gpu mark run the kernels themselves on CPU threads (oracle/fem2d_emu.cpp)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import build_host, fem2d_fast as Fz
from oracle.ref_harness.make_golden_fem2d import case_inputs

FEM2D_THREADS = 512
SMEM_OPTIN = 227 * 1024         # B200: shared memory one block may opt in to
GPU = torch.device("cuda:0")
# the bars: error relative to max|coeffs| (forward) and to max|reference gradient|
FWD_BAR, HOST_GRAD_BAR, FAST32_GRAD_BAR = 1e-5, 1e-5, 2e-4


# ---- restated from csrc/fem2d.cu: which CG template a mesh selects, and whether it fits in shared memory ----------
def rows_per_thread(N):
    need = (N + FEM2D_THREADS - 1) // FEM2D_THREADS
    return 1 if need <= 1 else (2 if need <= 2 else (4 if need <= 4 else 8))


def smem_bytes(N, T, D):
    al = lambda x: (x + 15) & ~15
    nbx = 4
    while nbx < 64 and 2 * nbx * nbx < T:
        nbx *= 2
    nb, rw = nbx * nbx, (D + 2 + 3) & ~3
    uni = max(al(rw * N * 8) + al(rw * N * 2), al((nb + 1) * 4) + al(nb * 4) + al(9 * T * 2))
    gauss_pre, star_rec, max_gauss = 72, 112, 16
    return (al(2 * N * 4) + al(T * 8) + 4 * al(N * 8) + al(2 * N * 8) + al(64 * 8) + al(16) + al(max_gauss * gauss_pre)
            + al(FEM2D_THREADS // 32 * D * star_rec) + uni)


# ---- meshes -------------------------------------------------------------------------------------------------------
def grid_mesh(nx, ny, jitter, seed):
    """nx x ny nodes on the unit square (node id = iy * nx + ix), every grid square split along its anti-diagonal
    (synth.unit_square_cells for nx != ny), interior nodes moved by up to jitter / 2 of the spacing."""
    xs, ys = np.linspace(0.0, 1.0, nx), np.linspace(0.0, 1.0, ny)
    X, Y = np.meshgrid(xs, ys, indexing="xy")
    pts = np.stack([X.ravel(), Y.ravel()], axis=1)
    ix, iy = np.meshgrid(np.arange(nx - 1), np.arange(ny - 1), indexing="xy")
    a = (iy * nx + ix).ravel()
    cells = np.stack([np.stack([a, a + 1, a + nx], 1), np.stack([a + 1, a + nx + 1, a + nx], 1)], 1).reshape(-1, 3)
    iix, iiy = np.arange(nx * ny) % nx, np.arange(nx * ny) // nx
    on_bc = (iix == 0) | (iix == nx - 1) | (iiy == 0) | (iiy == ny - 1)
    rng = np.random.default_rng(seed)
    pts[~on_bc] += (rng.random((int((~on_bc).sum()), 2)) - 0.5) * jitter / np.array([nx - 1, ny - 1])
    return cells.astype(np.int64), np.nonzero(on_bc)[0], pts.astype(np.float32)


def fan_mesh(M):
    """One interior vertex at (0.5, 0.5) -- a point of the 11 x 11 evaluation grid -- shared by M cells."""
    ang = np.arange(M) * 2 * np.pi / M + 0.1
    pts = np.concatenate([[[0.5, 0.5]], 0.5 + 0.45 * np.stack([np.cos(ang), np.sin(ang)], 1)]).astype(np.float32)
    cells = np.array([[0, 1 + k, 1 + (k + 1) % M] for k in range(M)], np.int64)
    return cells, np.arange(1, M + 1), pts


def gaussians(G, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.3, 0.7, size=(G, 2)), rng.uniform(0.2, 0.4, size=(G, 2))


def eval_grid(Q):
    x0 = torch.linspace(0, 1, Q)
    X, Y = torch.meshgrid(x0, x0, indexing="ij")
    return X.reshape(-1).numpy().copy(), Y.reshape(-1).numpy().copy()


def cotangent(sol, cen, scl, Q):
    """d mse(sol_b, u_true_b) / d sol_b for every mesh b: nonzero on every mesh, each against its own Gaussians."""
    ex, ey = eval_grid(Q)
    E = torch.stack([torch.from_numpy(ex), torch.from_numpy(ey)], -1)
    tgt = np.stack([Fz.u_true(E, torch.from_numpy(c), torch.from_numpy(s)).numpy() for c, s in zip(cen, scl)])
    return (2 * (sol - tgt) / (Q * Q)).astype(np.float32)


# ---- the kernels: on the GPU, or emulated on CPU threads -----------------------------------------------------------
def run_gpu(cells, bc, coords, cen, scl, K, Q):
    """coords [B, N, 2] fp32, cen / scl [B, G, 2] fp64 -> coeffs, sol, grad, CG iterations, cotangent (numpy)."""
    from g_adaptivity_b200 import fem2d
    N = coords.shape[1]
    topo = fem2d.Fem2DTopology(cells, bc, N, GPU)
    ex, ey = eval_grid(Q)
    xy = torch.from_numpy(coords).to(GPU).requires_grad_(True)
    sol, coeffs, iters = fem2d.fem2d_solve(xy, topo, torch.from_numpy(cen), torch.from_numpy(scl),
                                           torch.from_numpy(ex).to(GPU), torch.from_numpy(ey).to(GPU), K)
    g_sol = cotangent(sol.detach().cpu().numpy(), cen, scl, Q)
    sol.backward(torch.from_numpy(g_sol).to(GPU))
    return (coeffs.cpu().numpy(), sol.detach().cpu().numpy(), xy.grad.cpu().numpy(), iters.cpu().numpy(), g_sol)


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _tables(cells, bc, N):
    cells32 = np.ascontiguousarray(cells, dtype=np.int32)
    is_bc = np.zeros(N, np.uint8)
    is_bc[np.asarray(bc)] = 1
    sc_, sl_ = Fz.star_table(torch.as_tensor(cells, dtype=torch.long), N)
    return cells32, is_bc, sc_.numpy().astype(np.int32), sl_.numpy().astype(np.int32)


def run_emu(cells, bc, coords, cen, scl, K, Q):
    """run_gpu with k_fem2d_fwd / k_fem2d_bwd on CPU threads (oracle/fem2d_emu.cpp)."""
    lib = ctypes.CDLL(build_host.build_emu())
    B, N, _ = coords.shape
    cells32, is_bc, star_cell, star_loc = _tables(cells, bc, N)
    coords, cen, scl = (np.ascontiguousarray(coords, np.float32), np.ascontiguousarray(cen, np.float64),
                        np.ascontiguousarray(scl, np.float64))
    ex, ey = eval_grid(Q)
    coeffs, sol = np.zeros((B, N), np.float32), np.zeros((B, Q * Q), np.float32)
    grad, u64, iters = np.zeros((B, N, 2), np.float32), np.zeros((B, N), np.float64), np.zeros(B, np.int32)
    args = [_ptr(cells32), cells32.shape[0], _ptr(is_bc), N, _ptr(star_cell), _ptr(star_loc), star_cell.shape[1], _ptr(coords),
            _ptr(cen), _ptr(scl), cen.shape[1], B, int(K), _ptr(ex), _ptr(ey), Q * Q]
    assert lib.fem2d_emu(*args, None, _ptr(coeffs), _ptr(sol), _ptr(u64), None, _ptr(iters)) == 0
    g_sol = cotangent(sol, cen, scl, Q)
    assert lib.fem2d_emu(*args, _ptr(g_sol), _ptr(coeffs), _ptr(sol), _ptr(u64), _ptr(grad), None) == 0
    return coeffs, sol, grad, iters, g_sol


# ---- references, one mesh ------------------------------------------------------------------------------------------
def host_reference(cells, bc, pts, cen, scl, K, Q, g_sol):
    """The sequential host harness: coeffs, sol, grad, CG iterations (forward + adjoint)."""
    lib = ctypes.CDLL(build_host.build())
    N = pts.shape[0]
    cells32, is_bc, star_cell, star_loc = _tables(cells, bc, N)
    pts, cen, scl = np.ascontiguousarray(pts, np.float32), np.ascontiguousarray(cen, np.float64), np.ascontiguousarray(scl, np.float64)
    g_sol = np.ascontiguousarray(g_sol, np.float32)
    ex, ey = eval_grid(Q)
    coeffs, sol, grad = np.zeros(N, np.float32), np.zeros(Q * Q, np.float32), np.zeros((N, 2), np.float32)
    it = ctypes.c_int(0)
    assert lib.fem2d_host(_ptr(cells32), cells32.shape[0], _ptr(is_bc), N, _ptr(star_cell), _ptr(star_loc), star_cell.shape[1],
                          _ptr(pts), _ptr(cen), _ptr(scl), cen.shape[0], int(K), _ptr(ex), _ptr(ey), Q * Q, _ptr(g_sol),
                          _ptr(coeffs), _ptr(sol), _ptr(grad), ctypes.byref(it)) == 0
    return coeffs, sol, grad, it.value


def fast_reference(cells, bc, pts, cen, scl, K, Q, dtype, g_sol=None):
    """oracle/fem2d_fast.py in `dtype`: coeffs, sol and, given a cotangent, the autograd gradient."""
    ex, ey = eval_grid(Q)
    mesh = torch.from_numpy(pts).to(dtype).requires_grad_(g_sol is not None)
    X, Y = torch.from_numpy(ex).to(dtype), torch.from_numpy(ey).to(dtype)
    c, s = Fz.fem2d_fast(cells, bc, mesh, [X, Y], K, torch.from_numpy(cen), torch.from_numpy(scl))
    grad = None
    if g_sol is not None:
        s.reshape(-1).backward(torch.from_numpy(g_sol).to(dtype))
        grad = mesh.grad.numpy()
    return c.detach().reshape(-1).numpy(), s.detach().reshape(-1).numpy(), grad


def _rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - b).max() / np.abs(b).max())


def check_mesh(label, res, b, cells, bc, pts, cen, scl, K, Q, fast32=True, host_bar=HOST_GRAD_BAR):
    """Mesh b of a kernel run against the references; prints the observed errors."""
    coeffs, sol, grad, iters, g_sol = (r[b] for r in res)
    c64, s64, _ = fast_reference(cells, bc, pts, cen, scl, K, Q, torch.float64)
    scale = np.abs(c64).max()
    errs = {"coeffs": float(np.abs(coeffs - c64).max() / scale), "sol": float(np.abs(sol - s64).max() / scale)}
    _, _, g_host, _ = host_reference(cells, bc, pts, cen, scl, K, Q, g_sol)
    errs["grad_vs_host"] = _rel(grad, g_host)
    if fast32:
        _, _, g32 = fast_reference(cells, bc, pts, cen, scl, K, Q, torch.float32, g_sol)
        errs["grad_vs_fast32"] = _rel(grad, g32)
    print(f"[fem2d shapes] {label} mesh {b}: N={pts.shape[0]} K={K} Q={Q} G={cen.shape[0]} iters={int(iters)} "
          + " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    assert errs["coeffs"] <= FWD_BAR and errs["sol"] <= FWD_BAR, errs
    assert errs["grad_vs_host"] <= host_bar, errs
    assert errs.get("grad_vs_fast32", 0.0) <= FAST32_GRAD_BAR, errs
    assert 0 < iters < 20 * pts.shape[0]          # CG converged instead of stopping at its iteration cap


def batch_of(meshes, G, seed0):
    """Distinct per-mesh points and Gaussians stacked into a batch."""
    gs = [gaussians(G, seed0 + b) for b in range(len(meshes))]
    return (np.stack(meshes), np.stack([g[0] for g in gs]), np.stack([g[1] for g in gs]))


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_production_batch_of_distinct_meshes():
    """256 jittered 30x30 meshes (R = 2 CG template, 32 x 32 bin table, 10201 evaluation points: the point loop
    wraps 20 times), each with its own points, Gaussians and cotangent.  Four meshes against the references; every
    mesh against a launch of that mesh alone: bit for bit forward (no atomics decide a forward value), gradient to
    1e-6 (the backward accumulates in fp64 shared-memory atomics, whose order is not fixed)."""
    n, B, K, Q, G = 30, 256, 101, 101, 2
    cases = [case_inputs(n, G, 0.3, 1000 + b) for b in range(B)]
    cells, bc = cases[0][0], cases[0][1]
    assert rows_per_thread(n * n) == 2
    coords = np.stack([c[2] for c in cases])
    cen, scl = np.stack([c[3] for c in cases]), np.stack([c[4] for c in cases])
    res = run_gpu(cells, bc, coords, cen, scl, K, Q)
    coeffs, sol, grad, iters, g_sol = res
    assert np.all(iters > 0) and np.all(iters < 20 * n * n)
    assert np.all(np.abs(g_sol).max(axis=1) > 0) and np.all(np.abs(grad).max(axis=(1, 2)) > 0)
    for b in (0, 1, 127, 255):
        check_mesh("production 256 x 30x30", res, b, cells, bc, coords[b], cen[b], scl[b], K, Q)
    from g_adaptivity_b200 import fem2d
    topo = fem2d.Fem2DTopology(cells, bc, n * n, GPU)
    ex, ey = (torch.from_numpy(e).to(GPU) for e in eval_grid(Q))
    for b in range(B):
        xy = torch.from_numpy(coords[b:b + 1]).to(GPU).requires_grad_(True)
        s1, c1, it1 = fem2d.fem2d_solve(xy, topo, torch.from_numpy(cen[b:b + 1]), torch.from_numpy(scl[b:b + 1]), ex, ey, K)
        s1.backward(torch.from_numpy(g_sol[b:b + 1]).to(GPU))
        assert np.array_equal(c1.cpu().numpy()[0], coeffs[b]) and np.array_equal(s1.detach().cpu().numpy()[0], sol[b]), b
        assert int(it1[0]) == iters[b], b
        assert _rel(grad[b], xy.grad.cpu().numpy()[0]) <= 1e-6, b


# (nx, ny, rows per thread): node counts 512 / 513 and 1024 / 1025 on both sides of a template switch, and the
# largest square mesh whose shared memory fits (38 x 38 = 1444 nodes; N > 2048 would need R = 8 and does not fit)
CG_SHAPES = [(16, 32, 1), (19, 27, 2), (32, 32, 2), (25, 41, 4), (38, 38, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny,R", CG_SHAPES, ids=[f"{a}x{b}_R{r}" for a, b, r in CG_SHAPES])
def test_every_reachable_cg_template(nx, ny, R):
    N, K, Q = nx * ny, 101, 51
    cells, bc, _ = grid_mesh(nx, ny, 0.0, 0)
    assert rows_per_thread(N) == R
    assert smem_bytes(N, cells.shape[0], 6) <= SMEM_OPTIN
    if (nx, ny) == CG_SHAPES[-1][:2]:
        assert smem_bytes((nx + 1) ** 2, 2 * nx * nx, 6) > SMEM_OPTIN
    coords, cen, scl = batch_of([grid_mesh(nx, ny, 0.3, 10 + b)[2] for b in range(2)], 2, 20)
    res = run_gpu(cells, bc, coords, cen, scl, K, Q)
    for b in range(2):
        check_mesh(f"CG R={R} {nx}x{ny}", res, b, cells, bc, coords[b], cen[b], scl[b], K, Q)


def graded_mesh(n, seed):
    """Jittered n x n mesh mapped through x -> x^4 in both directions: cells shrink toward the corner (0, 0) down
    to (1 / (n - 1))^4 of the square, with large aspect ratios along the two sides that meet there."""
    cells, bc, pts = grid_mesh(n, n, 0.3, seed)
    return cells, bc, (pts.astype(np.float64) ** 4).astype(np.float32)


@pytest.mark.gpu
def test_graded_meshes():
    """The interior system of a graded 30x30 mesh has condition number 1.8e6 (370 for a jittered one).
    * fp32 fem2d_fast is no gradient reference here: its fp32 LU solve puts its gradient 1.9e-2 from the fp64
      evaluation of the same formulas, while the host harness (fp64 CG) is 5.7e-4 from it (tie decisions only).
    * Against the host harness the bar is 1e-4.  The GPU build may fuse the products of the triangle geometry
      (twice the signed area, the stiffness entries) into multiply-adds, which the host harness rounds
      separately, and this conditioning amplifies such rounding: on a B200 the gradient was 4e-6 and 3.3e-5 from
      the harness on the two meshes below, while the CPU emulation of the kernels, which rounds like the
      harness, is 2e-10 from it."""
    n, K, Q = 30, 101, 101
    cells, bc, _ = graded_mesh(n, 0)
    coords, cen, scl = batch_of([graded_mesh(n, 30 + b)[2] for b in range(2)], 2, 40)
    res = run_gpu(cells, bc, coords, cen, scl, K, Q)
    for b in range(2):
        check_mesh("graded x^4 30x30", res, b, cells, bc, coords[b], cen[b], scl[b], K, Q, fast32=False, host_bar=1e-4)


# K = 1 and 9: 3 Simpson points per side (9 per node: one partial batch of the backward's 3 x 32 points per lane
# round); K = 441: 21 per side (441 = 4 x 96 + 57: a partial final batch).  G = 1 and the limit G = 16.
QUAD_CASES = [(1, 2), (9, 2), (441, 2), (101, 1), (101, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("K,G", QUAD_CASES, ids=[f"K{k}_G{g}" for k, g in QUAD_CASES])
def test_quadrature_and_gaussian_limits(K, G):
    n, Q = 12, 41
    cells, bc, _ = grid_mesh(n, n, 0.0, 0)
    coords, cen, scl = batch_of([grid_mesh(n, n, 0.3, 50 + b)[2] for b in range(2)], G, 60)
    res = run_gpu(cells, bc, coords, cen, scl, K, Q)
    for b in range(2):
        check_mesh(f"K={K} G={G} 12x12", res, b, cells, bc, coords[b], cen[b], scl[b], K, Q)


@pytest.mark.gpu
def test_launch_limits_raise_before_launching():
    """17 Gaussians, a vertex of 17 cells and a mesh whose shared memory does not fit are refused by the host-side
    argument check with a RuntimeError -- directly and through GNN(loss_type='pde_loss')."""
    from g_adaptivity_b200 import fem2d

    def solve(cells, bc, pts, G):
        cen, scl = gaussians(G, 0)
        topo = fem2d.Fem2DTopology(cells, bc, pts.shape[0], GPU)
        ex, ey = (torch.from_numpy(e).to(GPU) for e in eval_grid(11))
        return fem2d.fem2d_solve(torch.from_numpy(pts[None]).to(GPU), topo, torch.from_numpy(cen[None]),
                                 torch.from_numpy(scl[None]), ex, ey, 9)

    cells, bc, pts = grid_mesh(8, 8, 0.3, 0)
    solve(cells, bc, pts, 16)
    with pytest.raises(RuntimeError, match=r"Gaussians .*\(got 17, 6\)"):
        solve(cells, bc, pts, 17)
    solve(*fan_mesh(16), 2)
    with pytest.raises(RuntimeError, match=r"cells per node \(got 2, 17\)"):
        solve(*fan_mesh(17), 2)
    cells, bc, pts = grid_mesh(39, 39, 0.3, 0)
    assert smem_bytes(39 * 39, cells.shape[0], 6) > SMEM_OPTIN
    with pytest.raises(RuntimeError, match="shared memory"):
        solve(cells, bc, pts, 2)
    torch.cuda.synchronize()

    from g_adaptivity_b200 import GNN, synth
    md, Q = (50, 50), 21
    ds = synth.SyntheticDataset(2, md, eval_quad_points=Q)
    data = synth.make_batch(md, 2, seed=0, eval_quad_points=Q)
    model = GNN(ds, synth.default_opt(md, device="cuda", loss_type="pde_loss", eval_quad_points=Q)).to("cuda")
    with pytest.raises(RuntimeError, match="shared memory"):
        model(data)


FAN_DEGREES = [12, 13, 16]


def _fan_case(M, runner):
    """The evaluation point on the vertex lies in all M cells of its star; every one of them is a hit, and the
    gradient of the hat function there averages over all of them."""
    cells, bc, pts = fan_mesh(M)
    K, Q = 101, 11
    ex, ey = eval_grid(Q)
    assert np.any((ex == pts[0, 0]) & (ey == pts[0, 1]))
    coords, cen, scl = batch_of([pts], 1, 70 + M)
    res = runner(cells, bc, coords, cen, scl, K, Q)
    check_mesh(f"fan M={M}", res, 0, cells, bc, pts, cen[0], scl[0], K, Q)


@pytest.mark.gpu
@pytest.mark.parametrize("M", FAN_DEGREES)
def test_vertex_of_many_cells_on_an_evaluation_point(M):
    _fan_case(M, run_gpu)


@pytest.mark.gpu
def test_repeated_meshes_agree():
    """The same mesh, Gaussians and cotangent at batch positions 0, 3 and 7 among distinct meshes.  The forward
    is bit for bit the same; the gradients agree to 1e-6 (fp64 shared-memory atomics: no fixed order)."""
    n, K, Q, B = 20, 101, 41, 8
    cells, bc, _ = grid_mesh(n, n, 0.0, 0)
    meshes = [grid_mesh(n, n, 0.3, 80 + b)[2] for b in range(B)]
    coords, cen, scl = batch_of(meshes, 2, 90)
    for b in (3, 7):
        coords[b], cen[b], scl[b] = coords[0], cen[0], scl[0]
    coeffs, sol, grad, iters, g_sol = run_gpu(cells, bc, coords, cen, scl, K, Q)
    assert np.array_equal(g_sol[3], g_sol[0]) and np.array_equal(g_sol[7], g_sol[0])
    for b in (3, 7):
        assert np.array_equal(coeffs[b], coeffs[0]) and np.array_equal(sol[b], sol[0]) and iters[b] == iters[0]
        assert _rel(grad[b], grad[0]) <= 1e-6
    assert not np.array_equal(coeffs[1], coeffs[0])


# ---- the same kernels emulated on CPU threads ------------------------------------------------------------------------
@pytest.mark.parametrize("M", FAN_DEGREES)
def test_emulated_vertex_of_many_cells_on_an_evaluation_point(M):
    _fan_case(M, run_emu)


def test_emulated_r2_template_at_the_production_shape():
    """One jittered 30x30 mesh at K = Q = 101: the R = 2 CG template, the 32 x 32 bin table and a point loop that
    wraps, against the host harness (which runs the same arithmetic sequentially) and fp64 fem2d_fast."""
    n, K, Q = 30, 101, 101
    cells, bc, pts, cen, scl = case_inputs(n, 2, 0.3, 7)
    assert rows_per_thread(n * n) == 2
    res = run_emu(cells, bc, pts[None], cen[None], scl[None], K, Q)
    check_mesh("emulated 30x30", res, 0, cells, bc, pts, cen, scl, K, Q, fast32=False)
