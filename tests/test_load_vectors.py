"""The load vectors the solvers build on the device, entry by entry against the oracle.

A wrong load vector gives a wrong answer, but the solution tests only see these vectors through a full solve on a small
grid, judged at 1e-8 relative L2, and never at the shapes where the fast paths branch: the plane chunks of the 3-D von
Mises projection (k_cell_vm + k_cell_gather), the grid-stride loops of the generic projection kernel (k_cell_rhs), the
P2 load of the cosine / sine initial condition (k_trig_table + k_p2_load) and the weighted assembly (k_weight_table +
k_wassemble).  The test entry points of include/pde_b200.h return each raw vector from the production launch.

CPU part: the windowed reference of the large von Mises cases against the full oracle.  GPU part (pytest.mark.gpu):
max|gpu - ref| <= BAR max|ref| on random (seeded) inputs, and two end-to-end cases that tie the entry points to the
tools.  The constant right-hand-side term of the stencil kernels is checked in test_gpu_parity.py
(test_operator_apply_matches_oracle) and at full size in test_steady_heat_with_end_temperatures_is_exactly_linear."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import fem_oracle as fo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# max|gpu - ref| <= BAR * max|ref|; worst measured on a B200 (1000 W): 2.5e-15 (k_p2_load, k_wassemble), von Mises
# 2.2e-15 (two-pass) / 2.3e-15 (k_cell_rhs<3>), k_cell_rhs<2> 1.8e-15, k_cell_rhs<1> 3.3e-16
BAR = 1e-12
E, NU = 210e9, 0.3


# ---------------------------------------------------------------- references
def cell_chunk(n):
    """Node planes per pass of the two-pass 3-D projection (launch_cell_rhs in csrc/kernels.cu)."""
    return min(max((48 << 20) // (n[0] * n[1]), 2), 32)


def box_axes(n, L):
    """BoxMesh vertex coordinates per axis on [0, L]: (i * L) / n."""
    return [(np.arange(k + 1, dtype=np.float64) * l) / float(k) for k, l in zip(n, L)]


def window_load(n, L, disp, lam, mu, quantity, box):
    """(vertex ids, load) of the 3-D von Mises projection on the vertices whose cells all lie in the cell box
    ((x0, x1), (y0, y1), (z0, z1)) or outside the grid: such a vertex sums the same simplices, with the same
    coordinates, in the sub-mesh of the box as in the full mesh.  A node plane p only touches the cell layers p - 1
    and p, so a few layers give the reference of a few planes of a grid the oracle cannot hold."""
    (x0, x1), (y0, y1), (z0, z1) = box
    sub = fo.box_mesh((0.0, 0.0, 0.0), (1.0, 1.0, 1.0), x1 - x0, y1 - y0, z1 - z0)
    ax = box_axes(n, L)
    Z, Y, X = np.meshgrid(ax[2][z0:z1 + 1], ax[1][y0:y1 + 1], ax[0][x0:x1 + 1], indexing="ij")
    sub.coords = np.stack([X.ravel(), Y.ravel(), Z.ravel()], axis=1)
    K = [k.ravel() for k in np.meshgrid(np.arange(z0, z1 + 1), np.arange(y0, y1 + 1), np.arange(x0, x1 + 1),
                                        indexing="ij")][::-1]
    gid = (K[2] * (n[1] + 1) + K[1]) * (n[0] + 1) + K[0]
    load = fo.cell_constant_load(sub, fo.von_mises_cells(sub, disp[gid], lam, mu, quantity))
    ok = np.ones(gid.size, dtype=bool)
    for k, (c0, c1), nc in zip(K, box, n):
        ok &= ((k - 1 < 0) | (k - 1 >= c0)) & ((k >= nc) | (k < c1))
    return gid[ok], load[ok]


def windowed_reference(n, L, disp, lam, mu, quantity, planes, tile=16):
    """window_load on the given node planes, over 3 x 3 tiles of tile x tile cells (both ends and the middle of x and
    y) per group of neighbouring planes; returns (vertex ids, load)."""
    nx, ny, nz = n
    spans = []
    for p in sorted(planes):
        lo, hi = max(p - 1, 0), min(p + 1, nz)
        if spans and lo <= spans[-1][1]:
            spans[-1][1] = max(spans[-1][1], hi)
        else:
            spans.append([lo, hi])
    xs = [(0, tile), (nx // 2 - tile // 2, nx // 2 + tile // 2), (nx - tile, nx)]
    ys = [(0, tile), (ny // 2 - tile // 2, ny // 2 + tile // 2), (ny - tile, ny)]
    ids, vals = [], []
    for z in spans:
        for x in xs:
            for y in ys:
                g, v = window_load(n, L, disp, lam, mu, quantity, (x, y, tuple(z)))
                keep = np.isin(g // ((nx + 1) * (ny + 1)), list(planes))
                ids.append(g[keep])
                vals.append(v[keep])
    ids, first = np.unique(np.concatenate(ids), return_index=True)
    return ids, np.concatenate(vals)[first]


def chunk_planes(n):
    """Node planes {0, 1, last} and the three around every chunk boundary of the two-pass projection."""
    nz, c = n[2], cell_chunk(n)
    planes = {0, 1, nz}
    for b in range(c, nz + 1, c):
        planes |= {b - 1, b, b + 1}
    return sorted(p for p in planes if p <= nz)


def projection_load_ref(dim, n, L, disp, quantity, plane_stress=True):
    """Oracle load of the projected stress / strain (1-D: E u' / u') of a displacement [nverts][dim]."""
    m = fo.make_mesh(dim, L, n)
    if dim == 1:
        _, G = fo._gradients(m)
        du = np.einsum("ca,ca->c", disp[:, 0][m.cells], G[:, :, 0])
        return fo.cell_constant_load(m, du if quantity == "strain" else E * du)
    lam, mu = fo.lame(E, NU, dim, plane_stress)
    return fo.cell_constant_load(m, fo.von_mises_cells(m, disp, lam, mu, quantity))


def dyadic(n):
    """Box lengths n h with one power-of-two spacing h for every axis (largest length in (1/2, 1]).  The oracle forms
    cell volumes and gradients from coordinate differences; with rounded coordinates those lose ~n eps, which would
    hide a kernel error of that size.  With h a power of two every coordinate and difference is exact."""
    h = 2.0 ** -int(np.ceil(np.log2(max(n))))
    return [k * h for k in n]


def random_disp(nv, dim, seed):
    return np.random.default_rng(seed).random((nv, dim)) - 0.5


def ratio_ok(tag, gpu, ref):
    ratio = np.abs(gpu - ref).max() / np.abs(ref).max()
    print(f"[load] {tag}: max|gpu-ref|/max|ref| = {ratio:.2e}")
    assert np.isfinite(gpu).all(), tag
    assert ratio <= BAR, (tag, ratio)


# ---------------------------------------------------------------- CPU: the windowed reference
@pytest.mark.parametrize("quantity", ["stress", "strain"])
def test_windowed_reference_equals_full_oracle(quantity):
    n, L = (10, 6, 40), (1.0, 0.6, 2.0)
    disp = random_disp(int(np.prod([k + 1 for k in n])), 3, 1)
    lam, mu = fo.lame(E, NU, 3)
    full = projection_load_ref(3, n, L, disp, quantity)
    planes = [0, 1, 12, 13, 14, 27, 40]
    ids, vals = windowed_reference(n, L, disp, lam, mu, quantity, planes, tile=4)
    nodes_per_plane = 11 * 7
    assert set(np.unique(ids // nodes_per_plane)) == set(planes)
    assert ids.size == len(planes) * nodes_per_plane    # at this size the overlapping tiles cover the planes
    assert np.abs(vals - full[ids]).max() <= 1e-14 * np.abs(full).max()
    # one full-plane window (a tile as wide as the grid) covers every vertex of its planes
    g, v = window_load(n, L, disp, lam, mu, quantity, ((0, 10), (0, 6), (19, 23)))
    assert set(np.unique(g // nodes_per_plane)) == {20, 21, 22}
    assert g.size == 3 * nodes_per_plane
    assert np.abs(v - full[g]).max() <= 1e-14 * np.abs(full).max()


@pytest.mark.parametrize("n", [(16, 8, 4), (9, 5, 7)])
def test_steady_source_solution_is_exact_at_the_nodes(n):
    """The closed form of test_steady_heat_with_end_temperatures_is_exactly_linear: T_left and T_right on the x-ends,
    natural side faces, source f: u = T_l + (T_r - T_l) x / L + f x (L - x) / (2 kappa) at the nodes."""
    L, kappa, f = (2.0, 0.7, 0.5), 1.7, 40.0
    ref = fo.solve_heat(3, L, n, kappa, steady=True, T_left=20.0, T_right=-5.0, source_type="constant",
                        source_value=f)
    x = ref.coords[:, 0]
    exact = 20.0 + (-5.0 - 20.0) * x / L[0] + f * x * (L[0] - x) / (2.0 * kappa)
    assert fo.rel_l2(ref.values[0], exact) <= 1e-12


def test_cell_chunk_and_chunk_planes():
    assert cell_chunk((1400, 1200, 40)) == 29 and cell_chunk((1280, 256, 256)) == 32
    assert cell_chunk((12, 7, 31)) == 32
    assert chunk_planes((12, 7, 33)) == [0, 1, 31, 32, 33]


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def P():
    import pde_solver_b200 as p
    return p


@pytest.fixture(scope="module")
def ctx(P):
    return P._lib.default_context()


def elast_params(P, dim, n, L, quantity, plane_stress=True, area=1.0):
    L_ = P._lib
    p = L_.ElastParams()
    p.dim = dim
    p.n = L_.i3(n)
    p.L = L_.d3(L)
    p.E, p.nu = E, NU
    p.body = L_.d3([0.0, 0.0, 0.0], 0.0)
    p.quantity = 1 if quantity == "strain" else 0
    p.plane_stress = 1 if plane_stress else 0
    p.area = float(area)
    return p


VM_FULL = [(12, 7, 31), (12, 7, 32), (12, 7, 33), (10, 9, 100), (128, 96, 40)]
VM_WINDOWED = [(1400, 1200, 40), (1280, 256, 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("n", VM_FULL + VM_WINDOWED)
def test_von_mises_load_3d(P, ctx, n):
    """k_cell_vm + k_cell_gather: one chunk, a last chunk of one and of two planes, four chunks, grid-striding cell
    passes, chunk = 29, and the benchmark grid (config 5, nine chunks)."""
    nv = int(np.prod([k + 1 for k in n]))
    disp = random_disp(nv, 3, sum(n))
    lam, mu = fo.lame(E, NU, 3)
    for q in ("stress", "strain"):
        load = P._lib.elast_projection_load(ctx, elast_params(P, 3, n, dyadic(n), q), disp)
        if n in VM_FULL:
            ref = projection_load_ref(3, n, dyadic(n), disp, q)
            ratio_ok(f"vm3d {n} {q}", load, ref)
        else:
            ids, ref = windowed_reference(n, dyadic(n), disp, lam, mu, q, chunk_planes(n))
            ratio_ok(f"vm3d {n} {q} planes {chunk_planes(n)}", load[ids], ref)


_SUB = r"""
import sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import pde_solver_b200 as P
from test_load_vectors import elast_params, dyadic
ctx = P._lib.default_context()
out = sys.argv[2]
for tag in sys.argv[3:]:
    nx, ny, nz, q = tag.split("_")
    n = (int(nx), int(ny), int(nz))
    disp = np.load(f"{out}/{nx}_{ny}_{nz}_disp.npy")
    np.save(f"{out}/{tag}_load.npy", P._lib.elast_projection_load(ctx, elast_params(P, 3, n, dyadic(n), q), disp))
"""


@pytest.mark.gpu
def test_generic_projection_kernel_3d(P, tmp_path):
    """k_cell_rhs<3>, the 3-D path behind PDE_B200_CELL_2PASS=0 (in a subprocess: the switch is read once)."""
    tags = []
    for n in [(12, 7, 33), (128, 96, 40)]:
        nv = int(np.prod([k + 1 for k in n]))
        np.save(tmp_path / ("%d_%d_%d_disp.npy" % n), random_disp(nv, 3, 7))
        tags += ["%d_%d_%d_%s" % (n + (q,)) for q in ("stress", "strain")]
    env = dict(os.environ, PDE_B200_CELL_2PASS="0")
    r = subprocess.run([sys.executable, "-c", _SUB, ROOT, str(tmp_path)] + tags, env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    for tag in tags:
        nx, ny, nz, q = tag.split("_")
        n = (int(nx), int(ny), int(nz))
        disp = np.load(tmp_path / f"{nx}_{ny}_{nz}_disp.npy")
        ratio_ok(f"cell_rhs<3> {tag}", np.load(tmp_path / f"{tag}_load.npy"),
                 projection_load_ref(3, n, dyadic(n), disp, q))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [(17, 9), (301, 2600)])
def test_projection_load_2d(P, ctx, n):
    """k_cell_rhs<2>: 301 x 2600 takes three ix passes of a 128-wide block and the grid-stride row loop."""
    L = dyadic(n)
    nv = (n[0] + 1) * (n[1] + 1)
    disp = random_disp(nv, 2, 3)
    for ps in (True, False):
        for q in ("stress", "strain"):
            load = P._lib.elast_projection_load(ctx, elast_params(P, 2, n, L, q, plane_stress=ps), disp)
            ratio_ok(f"cell_rhs<2> {n} plane_stress={ps} {q}", load, projection_load_ref(2, n, L, disp, q, ps))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [7, 100000])
def test_projection_load_1d(P, ctx, n):
    """k_cell_rhs<1>: axial strain u' (mode 2) and axial stress E u' (mode 3)."""
    disp = random_disp(n + 1, 1, 5)
    for q in ("stress", "strain"):
        load = P._lib.elast_projection_load(ctx, elast_params(P, 1, [n], dyadic([n]), q, area=2.0), disp)
        ratio_ok(f"cell_rhs<1> {n} {q}", load, projection_load_ref(1, [n], dyadic([n]), disp, q))


# ---------------------------------------------------------------- P2 load of the cosine / sine initial condition
AMP, KW = 3.0, 7.3
ORIGIN, SHIFTED = "origin", "shifted"


def trig_box(n, where):
    """(lo, hi): the box solvers' [0, L] or the cylinder branch's box shifted to y, z >= -1/2."""
    lo = [0.0, 0.0, 0.0] if where == ORIGIN else [0.0, -0.5, -0.5]
    return lo[:len(n)], [a + b for a, b in zip(lo, dyadic(n))]


@functools.lru_cache(maxsize=4)
def trig_mesh(dim, n, where):
    lo, hi = trig_box(n, where)
    if dim == 1:
        return fo.interval_mesh(n[0], lo[0], hi[0])
    if dim == 2:
        return fo.rectangle_mesh(lo[0], lo[1], hi[0], hi[1], n[0], n[1])
    return fo.box_mesh(lo, hi, *n)


@functools.lru_cache(maxsize=4)
def trig_load_ref(dim, n, where, kind):
    return fo.p2_load(trig_mesh(dim, n, where), fo._initial_expression(dim, kind, AMP, KW))


TRIG = [(1, (100000,), ORIGIN, "cosine"), (1, (100000,), ORIGIN, "sine"),
        (2, (301, 2600), ORIGIN, "cosine"), (2, (301, 2600), SHIFTED, "sine"),
        (3, (9, 5, 7), ORIGIN, "cosine"), (3, (9, 5, 7), ORIGIN, "sine"),
        (3, (9, 5, 7), SHIFTED, "cosine"), (3, (9, 5, 7), SHIFTED, "sine"),
        (3, (130, 50, 60), ORIGIN, "cosine"), (3, (130, 50, 60), SHIFTED, "sine")]


@pytest.mark.gpu
@pytest.mark.parametrize("dim,n,where,kind", TRIG)
def test_trig_initial_condition_load(P, ctx, dim, n, where, kind):
    """k_trig_table + k_p2_load, the right-hand side of project_trig_ic: the box solvers (lo = 0) and the shifted box
    of the cylinder branch."""
    lo, hi = trig_box(n, where)
    load = P._lib.trig_ic_load(ctx, dim, n, lo, hi, kind, AMP, KW)
    ratio_ok(f"p2_load {dim}d {n} {where} {kind}", load, trig_load_ref(dim, n, where, kind))


@pytest.mark.gpu
def test_trig_initial_condition_end_to_end(P):
    """values[0] of a 3-D cosine initial condition: the oracle mass solve of the P2 load (CG to 1e-14; LU does not
    fit at 400 k vertices), then the Dirichlet values."""
    n = (130, 50, 60)
    f = P._solve_heat_3d_raw(*dyadic(n), *n, 1.0, 2.5, 0.0, 0.01, 1, initial_type="cosine", initial_amplitude=AMP,
                             initial_wavenumber=KW, as_arrays=True)
    m = trig_mesh(3, n, ORIGIN)
    _, M = fo.assemble_stiffness_mass(m)
    b = trig_load_ref(3, n, ORIGIN, "cosine")
    d = M.diagonal()
    u, info = spla.cg(M, b, rtol=1e-14, atol=0.0, M=sp.diags(1.0 / d), maxiter=2000)
    assert info == 0
    dofs, vals = fo._merge_bcs(fo.heat_bcs(m, dyadic(n), T_boundary=2.5), m.nv)
    u[dofs] = vals
    err = fo.rel_l2(np.asarray(f.values)[0], u)
    print(f"[load] trig IC end to end {n}: rel L2 = {err:.2e}")
    assert err <= 1e-10, err


@pytest.mark.gpu
def test_elasticity_field_is_the_projection_of_its_displacement(P):
    """pde_elasticity_solve at 24 x 6 x 70 (three projection chunks): its field is the oracle projection of the
    displacement it returns."""
    from pde_solver_b200 import solvers
    n, L = (24, 6, 70), (1.0, 0.25, 3.0)
    m = fo.make_mesh(3, L, n)
    lam, mu = fo.lame(E, NU, 3)
    for q in ("stress", "strain"):
        _, val, disp = solvers._elasticity(3, L, n, E, NU, [1e4, -2e4, -76518.0], q, precond="gmg",
                                           want_displacement=True)
        ref, _ = fo.project_cell_constant(m, fo.von_mises_cells(m, disp, lam, mu, q))
        err = fo.rel_l2(val, ref)
        print(f"[load] elasticity end to end {n} {q}: rel L2 = {err:.2e}")
        assert err <= 1e-10, (q, err)


# ---------------------------------------------------------------- weighted assembly
OFFSETS = [(0, 0, 0), (1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1), (1, 1, 0), (-1, -1, 0),
           (1, 0, 1), (-1, 0, -1), (0, 1, 1), (0, -1, -1), (1, 1, 1), (-1, -1, -1)]


def stencil_of(A, n):
    """[nk][nverts] stencil of the assembled matrix A in the offset order of pde_wheat_level_coefs (internal axes; 2-D:
    x, z = user x, y) and the mask of entries whose neighbour lies in the grid."""
    dim = len(n)
    offs = {1: [o[:1] for o in OFFSETS[:3]], 2: [(o[0], o[2]) for o in OFFSETS if o[1] == 0], 3: OFFSETS}[dim]
    nn = np.array([k + 1 for k in n])
    xyz = np.indices(nn[::-1]).reshape(dim, -1)[::-1].T
    A = A.tocsr()
    out, inside = np.zeros((len(offs), xyz.shape[0])), np.zeros((len(offs), xyz.shape[0]), dtype=bool)
    for k, o in enumerate(offs):
        t = xyz + np.array(o)
        ok = np.all((t >= 0) & (t < nn), axis=1)
        j = sum(t[:, q] * int(np.prod(nn[:q])) for q in range(dim))
        rows = np.nonzero(ok)[0]
        out[k, rows] = np.asarray(A[rows, j[ok]]).ravel()
        inside[k] = ok
    assert np.isclose(np.abs(out).sum(), np.abs(A).sum(), rtol=1e-12)     # A has no entry outside the Kuhn stencil
    return out, inside


def weighted_case(P, name, n):
    """(WheatParams builder, oracle (K_w with the DG0 diffusivity, M_w, m_w)) of one weight of the tools at kappa 0.8,
    on a power-of-two box (dyadic) of the coordinate space: r from r_inner (0, or 1/8 for the hollow kinds), the
    cylinder centred on the x axis, the core box from the origin."""
    from pde_solver_b200 import solvers
    kappa = 0.8
    ext = dyadic(n)
    if name.startswith(("1d", "2d", "3d")):
        kind = name[:-len("_hollow")] if name.endswith("_hollow") else name
        dim, rpow, wsin, wdeg = solvers._CURVI[kind][:4]
        lo = [0.125 if name.endswith("_hollow") or dim == 3 else 0.0] + [0.0] * (dim - 1)
        weight, wkind, core = (rpow, wsin, wdeg), 0, None
        _, degree, wfun = fo.CURVILINEAR[kind]
    else:
        cyl = name.startswith("cylinder")
        lo = [0.0, -ext[1] / 2, -ext[2] / 2] if cyl else [0.0, 0.0, 0.0]
        weight, wkind = ((0, 0, 2), 1) if cyl else ((0, 0, 1), 0)
        rmax = min(ext[1], ext[2]) / (2 if cyl else 1)
        core = (0.6 * rmax, 8.0 if cyl else 25.0) if name.endswith("core") else None
        degree = 2 if cyl else 1
        wfun = (lambda x: np.sqrt(x[:, 1] ** 2 + x[:, 2] ** 2)) if cyl else (lambda x: np.ones(x.shape[0]))
    hi = [a + b for a, b in zip(lo, ext)]
    if len(n) == 1:
        mesh = fo.interval_mesh(n[0], lo[0], hi[0])
    elif len(n) == 2:
        mesh = fo.rectangle_mesh(lo[0], lo[1], hi[0], hi[1], n[0], n[1])
    else:
        mesh = fo.box_mesh(lo, hi, *n)
    kcell = np.full(mesh.cells.shape[0], kappa)
    if core is not None:
        X = mesh.coords[mesh.cells]
        rv = np.sqrt(X[:, :, 1] ** 2 + X[:, :, 2] ** 2)
        mid = X.mean(axis=1)
        kcell[(rv < core[0]).all(axis=1) & (np.sqrt(mid[:, 1] ** 2 + mid[:, 2] ** 2) < core[0])] = core[1]
    K, M, m = fo.assemble_weighted(mesh, wfun, degree, cell_scale=kcell)

    def params(steady, dt):
        return solvers._wheat_params(len(n), list(n), lo, hi, P._lib.make_bc({}), kappa, 0.0, dt, 1, steady, "constant",
                                     1.0, 1, weight=weight, weight_kind=wkind, core=core)
    return params, (K, M, m)


WEIGHTED = [("1d_cylindrical", (5001,)), ("1d_cylindrical_hollow", (5001,)), ("1d_spherical_hollow", (5001,)),
            ("2d_cylindrical_hollow", (301, 257)), ("2d_spherical", (301, 257)),
            ("3d_spherical", (33, 17, 21)), ("cylinder", (33, 17, 21)), ("core", (33, 17, 21)),
            ("cylinder_core", (33, 17, 21)), ("3d_spherical", (130, 50, 60)), ("cylinder_core", (130, 50, 60))]


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", WEIGHTED)
def test_weighted_assembly(P, ctx, name, n):
    """k_weight_table + k_wassemble: the full stencils of A = alpha M_w + beta K_w (steady: K_w with the
    diffusivity; transient: M_w + dt K_w) and of M_w, and the load m_w, on odd and ragged grids (the ones that run
    Jacobi-PCG on exactly this coefA)."""
    params, (K, M, m) = weighted_case(P, name, n)
    Mref, inside = stencil_of(M, n)
    Kref, _ = stencil_of(K, n)
    for steady, dt in ((True, 0.0), (False, 0.02)):
        cA, cM, load = P._lib.wheat_assembly(ctx, params(steady, dt))
        Aref = Kref if steady else Mref + dt * Kref
        tag = f"wassemble {name} {n} {'steady' if steady else 'transient'}"
        assert not cA[~inside].any() and not cM[~inside].any(), tag
        ratio_ok(tag + " coefA", cA, Aref)
        ratio_ok(tag + " coefM", cM, Mref)
        ratio_ok(tag + " load", load, m)
