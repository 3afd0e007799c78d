"""CPU oracle: NumPy/SciPy restatement of the FEniCS path of ziyu0425/PDE-Solver.

TEST INFRASTRUCTURE ONLY.  Nothing under ``pde_solver_b200/`` or ``fenics_mcp_server.py``
may import this file; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs do, and there only as the checker / CPU baseline.

PARITY UNPINNED: the reference has no tests, golden vectors or fixtures for this path
(SURVEY.md §4) and its arithmetic lives in FEniCS/DOLFIN 2019.1.0 + PETSc (conda-forge,
``requirements.txt:21-27``, ``Dockerfile:17-24``), which is not installable here.  This file
restates DOLFIN's published algorithms (mesh generators, P1 assembly, topological
DirichletBC, row-wise BC application + sparse direct LU, ``project``) and is pinned only by
closed-form known-answer tests (``tests/test_oracle.py``), not by reference outputs.

Reference call sites restated (all ``/root/reference/fenics_mcp_server.py``):
  IntervalMesh :229,1516   RectangleMesh :369,1648   BoxMesh :533,1803
  FunctionSpace/VectorFunctionSpace P1 :230,370,535,1649-1650,1804-1805
  DirichletBC + predicates :233-241, 373-376, 606-628, 1531-1534, 1681-1684, 1831-1834
  heat forms :261-262, 304-305, 393-394, 433-434, 657-658, 702-703
  solve(a == L, u, bcs) :265,311,397,440,661,709,1538,1688,1838  (default = sparse LU)
  initial conditions :276-297, 408-426, 672-691    time loop :309-318, 438-447, 707-716
  elasticity forms :1523-1528, 1653-1678, 1808-1828
  von Mises + project :1541-1546, 1691-1714, 1841-1862
"""
from __future__ import annotations

import itertools
import math
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

DOLFIN_EPS = 3.0e-16  # dolfin/common/constants.h; near(a,b) <=> |a-b| <= DOLFIN_EPS


def near(a, b, eps=DOLFIN_EPS):
    return np.abs(np.asarray(a) - b) <= eps


# --------------------------------------------------------------------------------------
# Mesh generators (DOLFIN 2019.1.0 IntervalMesh / RectangleMesh("right") / BoxMesh, serial)
# --------------------------------------------------------------------------------------

@dataclass
class Mesh:
    dim: int
    n: Tuple[int, int, int]           # cells per axis (0 for absent axes)
    coords: np.ndarray                # (nv, dim) float64
    cells_raw: np.ndarray             # (nc, dim+1) int32, generation order
    cells: np.ndarray                 # (nc, dim+1) int32, each row sorted ascending (mesh.order())
    lo: Tuple[float, ...] = ()
    hi: Tuple[float, ...] = ()

    @property
    def nv(self):
        return self.coords.shape[0]


def interval_mesh(nx: int, a: float, b: float) -> Mesh:
    """IntervalMesh(nx, a, b): x_i = a + ((b-a)/nx)*i ; cell i = (i, i+1)."""
    ab = (b - a) / float(nx)
    i = np.arange(nx + 1, dtype=np.float64)
    x = a + ab * i
    cells = np.stack([np.arange(nx), np.arange(nx) + 1], axis=1).astype(np.int32)
    return Mesh(1, (nx, 0, 0), x.reshape(-1, 1), cells, cells.copy(), (a,), (b,))


def rectangle_mesh(x0, y0, x1, y1, nx: int, ny: int) -> Mesh:
    """RectangleMesh(Point(x0,y0), Point(x1,y1), nx, ny, "right").

    x = x0 + ((x1-x0)/nx)*ix (spacing first, then multiply); vertex id = iy*(nx+1)+ix;
    per grid cell triangles (v0,v1,v3),(v0,v2,v3)."""
    ab = (x1 - x0) / float(nx)
    cd = (y1 - y0) / float(ny)
    xs = x0 + ab * np.arange(nx + 1, dtype=np.float64)
    ys = y0 + cd * np.arange(ny + 1, dtype=np.float64)
    X, Y = np.meshgrid(xs, ys, indexing="xy")  # Y varies along axis 0 -> iy slow
    coords = np.stack([X.ravel(), Y.ravel()], axis=1)
    ix, iy = np.meshgrid(np.arange(nx), np.arange(ny), indexing="xy")
    v0 = (iy * (nx + 1) + ix).ravel()
    v1 = v0 + 1
    v2 = v0 + (nx + 1)
    v3 = v1 + (nx + 1)
    cells = np.empty((2 * nx * ny, 3), dtype=np.int64)
    cells[0::2] = np.stack([v0, v1, v3], axis=1)
    cells[1::2] = np.stack([v0, v2, v3], axis=1)
    cells = cells.astype(np.int32)
    return Mesh(2, (nx, ny, 0), coords, cells, np.sort(cells, axis=1), (x0, y0), (x1, y1))


BOX_TETS = ((0, 1, 3, 7), (0, 1, 7, 5), (0, 5, 7, 4), (0, 3, 2, 7), (0, 6, 4, 7), (0, 2, 6, 7))


def box_mesh(p0, p1, nx: int, ny: int, nz: int) -> Mesh:
    """BoxMesh(Point(p0), Point(p1), nx, ny, nz).

    x = a + ix*(b-a)/nx evaluated as a + ((ix*(b-a))/nx) (C++ precedence); vertex id =
    iz*(nx+1)*(ny+1) + iy*(nx+1) + ix; six tetrahedra per grid cell sharing diagonal v0-v7."""
    a, c, e = (float(v) for v in p0)
    b, d, f = (float(v) for v in p1)
    xs = a + (np.arange(nx + 1, dtype=np.float64) * (b - a)) / float(nx)
    ys = c + (np.arange(ny + 1, dtype=np.float64) * (d - c)) / float(ny)
    zs = e + (np.arange(nz + 1, dtype=np.float64) * (f - e)) / float(nz)
    Z, Y, X = np.meshgrid(zs, ys, xs, indexing="ij")
    coords = np.stack([X.ravel(), Y.ravel(), Z.ravel()], axis=1)
    iz, iy, ix = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    v0 = (iz * (nx + 1) * (ny + 1) + iy * (nx + 1) + ix).ravel().astype(np.int64)
    v = [v0, v0 + 1, v0 + (nx + 1), v0 + 1 + (nx + 1)]
    v = v + [w + (nx + 1) * (ny + 1) for w in v]
    cells = np.empty((6 * v0.size, 4), dtype=np.int64)
    for t, tet in enumerate(BOX_TETS):
        cells[t::6] = np.stack([v[k] for k in tet], axis=1)
    cells = cells.astype(np.int32)
    return Mesh(3, (nx, ny, nz), coords, cells, np.sort(cells, axis=1), (a, c, e), (b, d, f))


def make_mesh(dim: int, L: Sequence[float], n: Sequence[int]) -> Mesh:
    if dim == 1:
        return interval_mesh(n[0], 0.0, L[0])
    if dim == 2:
        return rectangle_mesh(0.0, 0.0, L[0], L[1], n[0], n[1])
    return box_mesh((0.0, 0.0, 0.0), tuple(L[:3]), n[0], n[1], n[2])


# --------------------------------------------------------------------------------------
# DOF maps (SURVEY appendix A.3).  Natural numbering == parameters["reorder_dofs_serial"]=False
# --------------------------------------------------------------------------------------

def cell_dofs_scalar(mesh: Mesh) -> np.ndarray:
    """P1 scalar: one dof per vertex, dof == vertex index (UFC numbering)."""
    return mesh.cells.copy()


def cell_dofs_vector(mesh: Mesh, ncomp: int, layout: str = "blocked") -> np.ndarray:
    """Vector P1 cell dofs, (nc, ncomp*(d+1)), component-major within a cell as in UFC.

    layout 'blocked'     : dof = c*nv + v   (UFC / reorder off)
    layout 'interleaved' : dof = ncomp*v + c (block size ncomp, what reordering produces)"""
    c = mesh.cells.astype(np.int64)
    out = []
    for comp in range(ncomp):
        out.append(comp * mesh.nv + c if layout == "blocked" else ncomp * c + comp)
    return np.concatenate(out, axis=1).astype(np.int32)


# --------------------------------------------------------------------------------------
# Boundary facets and topological DirichletBC (SURVEY appendix A.4)
# --------------------------------------------------------------------------------------

def exterior_facets(mesh: Mesh) -> np.ndarray:
    """(nf, d) vertex ids of facets that belong to exactly one cell."""
    d = mesh.dim
    c = mesh.cells.astype(np.int64)
    facets = np.concatenate([np.delete(c, k, axis=1) for k in range(d + 1)], axis=0)
    facets = np.sort(facets, axis=1)
    uniq, counts = np.unique(facets, axis=0, return_counts=True)
    return uniq[counts == 1]


def dirichlet_dofs(mesh: Mesh, predicate: Callable[[np.ndarray, bool], np.ndarray]) -> np.ndarray:
    """DirichletBC(V, g, predicate), method='topological': exterior facets whose vertices AND
    midpoint all satisfy predicate(x, on_boundary=True); returns sorted vertex ids."""
    f = exterior_facets(mesh)
    X = mesh.coords[f]                       # (nf, d, dim)
    ok = np.ones(f.shape[0], dtype=bool)
    for k in range(f.shape[1]):
        ok &= predicate(X[:, k, :], True)
    ok &= predicate(X.mean(axis=1), True)
    return np.unique(f[ok].ravel())


# --------------------------------------------------------------------------------------
# P1 element matrices and assembly
# --------------------------------------------------------------------------------------

def _gradients(mesh: Mesh):
    """Per cell: volume (nc,) and basis gradients G (nc, d+1, d)."""
    d = mesh.dim
    X = mesh.coords[mesh.cells]                      # (nc, d+1, d)
    E = X[:, 1:, :] - X[:, :1, :]                    # rows e_a = x_a - x_0
    det = np.linalg.det(E)
    vol = np.abs(det) / math.factorial(d)
    Einv = np.linalg.inv(E)                          # columns = grad phi_a, a=1..d
    G = np.empty((X.shape[0], d + 1, d))
    G[:, 1:, :] = np.transpose(Einv, (0, 2, 1))
    G[:, 0, :] = -G[:, 1:, :].sum(axis=1)
    return vol, G


def _assemble(rows, cols, vals, n) -> sp.csr_matrix:
    A = sp.coo_matrix((vals.ravel(), (rows.ravel(), cols.ravel())), shape=(n, n)).tocsr()
    A.sum_duplicates()
    return A


def assemble_stiffness_mass(mesh: Mesh) -> Tuple[sp.csr_matrix, sp.csr_matrix]:
    """K_ij = ∫ ∇φ_i·∇φ_j (degree-0 quadrature exact), M_ij = ∫ φ_i φ_j (exact)."""
    d = mesh.dim
    vol, G = _gradients(mesh)
    Ke = vol[:, None, None] * np.einsum("cai,cbi->cab", G, G)
    Me = vol[:, None, None] / ((d + 1) * (d + 2)) * (np.ones((d + 1, d + 1)) + np.eye(d + 1))[None]
    c = mesh.cells.astype(np.int64)
    rows = np.repeat(c[:, :, None], d + 1, axis=2)
    cols = np.repeat(c[:, None, :], d + 1, axis=1)
    return _assemble(rows, cols, Ke, mesh.nv), _assemble(rows, cols, Me, mesh.nv)


def assemble_elasticity(mesh: Mesh, lam: float, mu: float) -> sp.csr_matrix:
    """a(u,v) = ∫ σ(u):ε(v), σ = λ tr(ε) I + 2μ ε.  Interleaved dofs: d*vertex + comp.

    K[(a,i),(b,j)] = |c| (λ ∂iφa ∂jφb + μ ∂jφa ∂iφb + μ δij ∇φa·∇φb)."""
    d = mesh.dim
    vol, G = _gradients(mesh)
    GG = np.einsum("cak,cbk->cab", G, G)
    Ke = (lam * np.einsum("cai,cbj->caibj", G, G)
          + mu * np.einsum("caj,cbi->caibj", G, G)
          + mu * np.einsum("cab,ij->caibj", GG, np.eye(d)))
    Ke *= vol[:, None, None, None, None]
    c = mesh.cells.astype(np.int64)
    dof = d * c[:, :, None] + np.arange(d)[None, None, :]          # (nc, d+1, d)
    nd = (d + 1) * d
    dof = dof.reshape(-1, nd)
    rows = np.repeat(dof[:, :, None], nd, axis=2)
    cols = np.repeat(dof[:, None, :], nd, axis=1)
    return _assemble(rows, cols, Ke.reshape(-1, nd, nd), d * mesh.nv)


def lumped_load(mesh: Mesh) -> np.ndarray:
    """m_i = ∫ φ_i = Σ_{cells ∋ i} |c|/(d+1)."""
    vol, _ = _gradients(mesh)
    m = np.zeros(mesh.nv)
    np.add.at(m, mesh.cells.ravel(), np.repeat(vol / (mesh.dim + 1), mesh.dim + 1))
    return m


def apply_bc_rowwise(A: sp.csr_matrix, b: np.ndarray, dofs: np.ndarray, vals: np.ndarray):
    """DirichletBC.apply(A, b): BC rows zeroed, diagonal 1, b_i = g (columns untouched)."""
    A = A.tolil(copy=True) if A.shape[0] < 2000 else A.tocsr(copy=True)
    if sp.issparse(A) and A.format == "lil":
        for i in dofs:
            A.rows[i] = [int(i)]
            A.data[i] = [1.0]
        A = A.tocsr()
    else:
        keep = np.ones(A.shape[0])
        keep[dofs] = 0.0
        A = sp.diags(keep) @ A
        diag = np.zeros(A.shape[0])
        diag[dofs] = 1.0
        A = (A + sp.diags(diag)).tocsr()
    b = b.copy()
    b[dofs] = vals
    return A, b


def apply_bc_symmetric(A: sp.csr_matrix, b: np.ndarray, dofs: np.ndarray, vals: np.ndarray):
    """Symmetric elimination (what a CG solver needs); same solution as the row-wise form."""
    n = A.shape[0]
    g = np.zeros(n)
    g[dofs] = vals
    b2 = b - A @ g
    keep = np.ones(n)
    keep[dofs] = 0.0
    Dk = sp.diags(keep)
    diag = np.zeros(n)
    diag[dofs] = 1.0
    A2 = (Dk @ A @ Dk + sp.diags(diag)).tocsr()
    b2[dofs] = vals
    return A2, b2


def _row_scale(A: sp.csr_matrix):
    """1/max|row|: DOLFIN's row-wise BC rows carry a bare 1.0 next to O(E) ~ 1e11 stiffness rows;
    SuperLU then leaves ~1e-10 absolute error on the clamped dofs (1e-5 relative in u).  Scaling
    rows does not change the solution A^-1 b, only the rounding (UMFPACK/MUMPS, which the
    reference's PETSc LU uses, scale rows by default)."""
    s = np.asarray(abs(A).max(axis=1).todense()).ravel()
    s[s == 0] = 1.0
    return 1.0 / s


class _ScaledLU:
    def __init__(self, A: sp.csr_matrix):
        self.s = _row_scale(A)
        self.lu = spla.splu((sp.diags(self.s) @ A).tocsc())

    def solve(self, b):
        return self.lu.solve(self.s * b)


def lu_solve(A: sp.csr_matrix, b: np.ndarray) -> np.ndarray:
    return _ScaledLU(A.tocsr()).solve(b)


# --------------------------------------------------------------------------------------
# project(Expression(..., degree=2), V)  (SURVEY appendix A.5)
# --------------------------------------------------------------------------------------

def project_p2_expression(mesh: Mesh, fn: Callable[[np.ndarray], np.ndarray]) -> np.ndarray:
    """project(Expression(degree=2), P1): the P2 load of p2_load, then the consistent-mass system with LU."""
    _, M = assemble_stiffness_mass(mesh)
    return lu_solve(M, p2_load(mesh, fn))


def p2_load(mesh: Mesh, fn: Callable[[np.ndarray], np.ndarray]) -> np.ndarray:
    """b_i = ∫ I_P2(fn) φ_i: fn interpolated into P2 on every cell (vertices + edge midpoints) and integrated
    exactly against P1."""
    d = mesh.dim
    vol, _ = _gradients(mesh)
    c = mesh.cells.astype(np.int64)
    X = mesh.coords[c]
    fac = math.factorial
    # ∫ λ^α = |c| d! α! / (d+|α|)!
    I = lambda *al: fac(d) * np.prod([fac(a) for a in al]) / fac(d + sum(al))
    vself = 2 * I(3) - I(2)            # ∫ λa(2λa-1) λa
    voth = 2 * I(2, 1) - I(1, 1)       # ∫ λa(2λa-1) λi, i != a
    ein = 4 * I(2, 1)                  # ∫ 4 λa λb λi, i in {a,b}
    eout = 4 * I(1, 1, 1) if d >= 2 else 0.0
    b = np.zeros(mesh.nv)
    fv = fn(X.reshape(-1, d)).reshape(c.shape)                       # vertex values
    for i in range(d + 1):
        contrib = np.zeros(c.shape[0])
        for a in range(d + 1):
            contrib += fv[:, a] * (vself if a == i else voth)
        for a, bb in itertools.combinations(range(d + 1), 2):
            fm = fn(0.5 * (X[:, a, :] + X[:, bb, :]))
            contrib += fm * (ein if i in (a, bb) else eout)
        np.add.at(b, c[:, i], contrib * vol)
    return b


# --------------------------------------------------------------------------------------
# Heat solvers: _solve_heat_{1,2,3}d_raw restated (box / uniform-κ branches)
# --------------------------------------------------------------------------------------

@dataclass
class Field:
    coords: np.ndarray     # (N, 3)
    values: np.ndarray     # (Nt, N)
    times: np.ndarray      # (Nt,)
    dim: int
    meta: Dict[str, object] = field(default_factory=dict)
    aux: Dict[str, object] = field(default_factory=dict)


def heat_bcs(mesh: Mesh, L, T_boundary=0.0, T_left=None, T_right=None, T_side=None):
    """List of (dofs, value) in the order the reference builds its bcs list.

    1D (:233-241): [left, right].  2D (:373-376): [all].  3D (:576-628): directional
    [left, right, other_faces] if any of T_left/T_right/T_side is given, else [all]."""
    Lx = L[0]
    left = lambda x, ob: near(x[:, 0], 0.0)
    right = lambda x, ob: near(x[:, 0], Lx)
    allb = lambda x, ob: np.ones(x.shape[0], dtype=bool)
    other = lambda x, ob: ~(near(x[:, 0], 0.0) | near(x[:, 0], Lx))
    if mesh.dim == 1:
        return [(dirichlet_dofs(mesh, left), float(T_left)), (dirichlet_dofs(mesh, right), float(T_right))]
    if mesh.dim == 3 and (T_left is not None or T_right is not None or T_side is not None):
        out = []
        if T_left is not None:
            out.append((dirichlet_dofs(mesh, left), float(T_left)))
        if T_right is not None:
            out.append((dirichlet_dofs(mesh, right), float(T_right)))
        if T_side is not None:
            out.append((dirichlet_dofs(mesh, other), float(T_side)))
        return out
    return [(dirichlet_dofs(mesh, allb), float(T_boundary))]


def _merge_bcs(bcs, n):
    """Later BCs win on shared dofs (list order, as bc.apply is called in sequence)."""
    g = np.full(n, np.nan)
    for dofs, val in bcs:
        g[dofs] = val
    dofs = np.nonzero(~np.isnan(g))[0]
    return dofs, g[dofs]


def _initial_expression(dim, kind, A, k):
    f = np.cos if kind == "cosine" else np.sin

    def fn(x):
        out = A * f(k * x[:, 0])
        for ax in range(1, dim):
            out = out * f(k * x[:, ax])
        return out
    return fn


def solve_heat(dim: int, L: Sequence[float], n: Sequence[int], diffusivity: float,
               T_initial: float = 0.0, dt: float = 0.01, num_steps: int = 50,
               T_boundary: float = 0.0, T_left=None, T_right=None, T_side=None,
               steady: bool = False, source_type: str = "none", source_value: float = 0.0,
               initial_type: str = "constant", initial_amplitude: float = 1.0,
               initial_wavenumber: float = 1.0, symmetric: bool = False) -> Field:
    """Backward-Euler / steady P1 heat solve, `_solve_heat_{1,2,3}d_raw` (:204-338, 345-468,
    475-762 box branch).  Output in natural dof order (1D: sorted by x, which is the same)."""
    mesh = make_mesh(dim, L, n)
    K, M = assemble_stiffness_mass(mesh)
    m = lumped_load(mesh)
    bcs = heat_bcs(mesh, L, T_boundary, T_left, T_right, T_side)
    bc_dofs, bc_vals = _merge_bcs(bcs, mesh.nv)
    f = float(source_value) if source_type == "constant" else 0.0
    kappa = float(diffusivity)
    apply_bc = apply_bc_symmetric if symmetric else apply_bc_rowwise
    snaps, times = [], []
    if steady:
        A, b = apply_bc(kappa * K, f * m, bc_dofs, bc_vals)
        snaps.append(lu_solve(A, b))
        times.append(0.0)
    else:
        if initial_type == "zero":
            u = np.zeros(mesh.nv)
        elif initial_type in ("cosine", "sine"):
            u = project_p2_expression(mesh, _initial_expression(dim, initial_type, initial_amplitude,
                                                                initial_wavenumber))
        else:
            u = np.full(mesh.nv, float(T_initial))
        u[bc_dofs] = bc_vals
        snaps.append(u.copy())
        times.append(0.0)
        A0 = (M + (dt * kappa) * K).tocsr()
        A, _ = apply_bc(A0, np.zeros(mesh.nv), bc_dofs, bc_vals)
        lu = _ScaledLU(A.tocsr())
        for step in range(num_steps):
            b = M @ u + (dt * f) * m
            if symmetric:
                _, b = apply_bc_symmetric(A0, b, bc_dofs, bc_vals)
            else:
                b[bc_dofs] = bc_vals
            u = lu.solve(b)
            snaps.append(u.copy())
            times.append((step + 1) * dt)
    coords = np.zeros((mesh.nv, 3))
    coords[:, :dim] = mesh.coords
    return Field(coords, np.array(snaps), np.array(times), dim,
                 aux={"mesh": mesh, "bc_dofs": bc_dofs, "bc_vals": bc_vals})


# --------------------------------------------------------------------------------------
# Elasticity solvers: _solve_elasticity_{1,2,3}d_static restated
# --------------------------------------------------------------------------------------

def lame(E: float, nu: float, dim: int, plane_stress: bool = True):
    """3D / plane strain (:1813-1814, 1664-1665); 2D plane stress λ = Eν/(1-ν²) (:1660-1661)."""
    mu = E / (2.0 * (1.0 + nu))
    if dim == 2 and plane_stress:
        lam = E * nu / (1.0 - nu ** 2)
    else:
        lam = E * nu / ((1.0 + nu) * (1.0 - 2.0 * nu))
    return lam, mu


def von_mises_cells(mesh: Mesh, u: np.ndarray, lam: float, mu: float, quantity: str) -> np.ndarray:
    """Cell-wise constant equivalent stress/strain (:1691-1711, 1841-1859).  u is (nv, d).
    The deviator uses 1/3 in every dimension (quirk kept: 2D uses 1/3 with a 2x2 identity)."""
    d = mesh.dim
    _, G = _gradients(mesh)
    gu = np.einsum("cai,cak->cik", u[mesh.cells], G)         # ∂k u_i
    eps = 0.5 * (gu + np.transpose(gu, (0, 2, 1)))
    I = np.eye(d)[None]
    tr_e = np.trace(eps, axis1=1, axis2=2)[:, None, None]
    if quantity == "strain":
        dev = eps - (1.0 / 3.0) * tr_e * I
        return np.sqrt(2.0 / 3.0 * np.einsum("cij,cij->c", dev, dev))
    sig = lam * tr_e * I + 2.0 * mu * eps
    tr_s = np.trace(sig, axis1=1, axis2=2)[:, None, None]
    dev = sig - (1.0 / 3.0) * tr_s * I
    return np.sqrt(3.0 / 2.0 * np.einsum("cij,cij->c", dev, dev))


def project_cell_constant(mesh: Mesh, vc: np.ndarray) -> np.ndarray:
    """project(v, P1) for a cell-wise constant v: M x = cell_constant_load(mesh, v), LU (appendix A.5)."""
    b = cell_constant_load(mesh, vc)
    _, M = assemble_stiffness_mass(mesh)
    return lu_solve(M, b), b


def cell_constant_load(mesh: Mesh, vc: np.ndarray) -> np.ndarray:
    """b_i = Σ_{c ∋ i} v_c |c|/(d+1): the load of project(v, P1) for a cell-wise constant v."""
    vol, _ = _gradients(mesh)
    b = np.zeros(mesh.nv)
    np.add.at(b, mesh.cells.ravel(), np.repeat(vc * vol / (mesh.dim + 1), mesh.dim + 1))
    return b


def solve_elasticity(dim: int, L: Sequence[float], n: Sequence[int], E: float, nu: float = 0.3,
                     body: Sequence[float] = (0.0, 0.0, 0.0), quantity: str = "stress",
                     plane_stress: bool = True, area: float = 1.0, symmetric: bool = False) -> Field:
    """Static P1 elasticity clamped at x=0 with constant body force, then the projected scalar.

    1D (:1470-1587): EA u'' = -f, output project(u') or project(E u').
    2D/3D (:1593-1743, 1749-1892): vector P1, von Mises, project to scalar P1."""
    mesh = make_mesh(dim, L, n)
    left = lambda x, ob: near(x[:, 0], 0.0)
    clamp = dirichlet_dofs(mesh, left)
    apply_bc = apply_bc_symmetric if symmetric else apply_bc_rowwise
    coords = np.zeros((mesh.nv, 3))
    coords[:, :dim] = mesh.coords
    if dim == 1:
        K, _ = assemble_stiffness_mass(mesh)
        A, b = apply_bc((E * area) * K, float(body[0]) * lumped_load(mesh), clamp, np.zeros(clamp.size))
        u = lu_solve(A, b)
        _, G = _gradients(mesh)
        du = np.einsum("ca,ca->c", u[mesh.cells], G[:, :, 0])
        vc = du if quantity == "strain" else E * du
        val, rhs = project_cell_constant(mesh, vc)
        return Field(coords, val[None, :], np.array([0.0]), 1, aux={"mesh": mesh, "u": u[:, None], "cell": vc})
    lam, mu = lame(E, nu, dim, plane_stress)
    A0 = assemble_elasticity(mesh, lam, mu)
    m = lumped_load(mesh)
    b0 = (m[:, None] * np.asarray(body[:dim], dtype=float)[None, :]).ravel()
    dofs = (dim * clamp[:, None] + np.arange(dim)[None, :]).ravel()
    A, b = apply_bc(A0, b0, dofs, np.zeros(dofs.size))
    u = lu_solve(A, b).reshape(-1, dim)
    vc = von_mises_cells(mesh, u, lam, mu, quantity)
    val, rhs = project_cell_constant(mesh, vc)
    return Field(coords, val[None, :], np.array([0.0]), dim,
                 aux={"mesh": mesh, "u": u, "cell": vc, "lam": lam, "mu": mu, "rhs": rhs, "A": A0, "b": b0,
                      "clamp": clamp})


# --------------------------------------------------------------------------------------
# Parity metric (SURVEY §8c): canonicalise by lattice index recovered from coordinates
# --------------------------------------------------------------------------------------

def canonical_order(coords: np.ndarray, L: Sequence[float], n: Sequence[int]) -> np.ndarray:
    """Permutation that sorts dofs into natural lattice order (x fastest) from their coordinates,
    so an L2 comparison is independent of any dof renumbering."""
    idx = np.zeros(coords.shape[0], dtype=np.int64)
    stride = 1
    for ax in range(3):
        if ax < len(n) and n[ax] > 0:
            i = np.rint(coords[:, ax] / (L[ax] / n[ax])).astype(np.int64)
            idx += i * stride
            stride *= n[ax] + 1
    return np.argsort(idx, kind="stable")


def rel_l2(a: np.ndarray, b: np.ndarray) -> float:
    nb = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / nb) if nb > 0 else float(np.linalg.norm(a - b))


# --------------------------------------------------------------------------------------
# Curvilinear heat tools (reference :769-1464): the same P1 backward-Euler loop with ONE scalar weight w(x) in
# every term,  a = w u v dx + dt k w grad(u).grad(v) dx,  L = w u_n v dx + dt w f v dx,  where w is an
# Expression of degree 1 (x[0]) or 2 (x[0]^2, x[0]^2 sin(x[1])).  FFC interpolates a degree-p Expression into
# the P_p element on every cell and integrates the resulting polynomial exactly, which is what is restated.
# --------------------------------------------------------------------------------------

def _mono(d, alpha):
    """Integral of prod(lambda_k^alpha_k) over the unit-volume d-simplex: d! prod(alpha!) / (d + |alpha|)!"""
    f = math.factorial
    return f(d) * np.prod([f(a) for a in alpha]) / f(d + sum(alpha))


def _weight_basis_integrals(d, degree):
    """Per weight basis function k: (Ws[k] = int psi_k, Wl[k][i] = int psi_k lam_i, Wm[k][i][j] = int psi_k lam_i lam_j),
    all for a unit-volume simplex; weight basis = P1 (vertices) or P2 (vertices, then edges a<b)."""
    nv = d + 1

    def e(*idx):
        a = [0] * nv
        for i in idx:
            a[i] += 1
        return a

    polys = []   # each psi as a list of (coef, exponent-vector)
    for v in range(nv):
        if degree == 1:
            polys.append([(1.0, e(v))])
        else:
            polys.append([(2.0, e(v, v)), (-1.0, e(v))])
    if degree == 2:
        for a, b in itertools.combinations(range(nv), 2):
            polys.append([(4.0, e(a, b))])
    nk = len(polys)
    Ws, Wl, Wm = np.zeros(nk), np.zeros((nk, nv)), np.zeros((nk, nv, nv))
    for k, poly in enumerate(polys):
        for cf, ex in poly:
            Ws[k] += cf * _mono(d, ex)
            for i in range(nv):
                exi = list(ex)
                exi[i] += 1
                Wl[k, i] += cf * _mono(d, exi)
                for j in range(nv):
                    exij = list(exi)
                    exij[j] += 1
                    Wm[k, i, j] += cf * _mono(d, exij)
    return Ws, Wl, Wm


def assemble_weighted(mesh: Mesh, wfun: Callable[[np.ndarray], np.ndarray], degree: int, cell_scale=None):
    """(Kw, Mw, mw): int I_p(w) grad(phi_i).grad(phi_j), int I_p(w) phi_i phi_j, int I_p(w) phi_i.
    cell_scale: optional per-cell factor of the stiffness term only (a DG0 diffusivity)."""
    d = mesh.dim
    vol, G = _gradients(mesh)
    c = mesh.cells.astype(np.int64)
    X = mesh.coords[c]
    nv = d + 1
    Ws, Wl, Wm = _weight_basis_integrals(d, degree)
    wk = [wfun(X[:, a, :]) for a in range(nv)]
    if degree == 2:
        wk += [wfun(0.5 * (X[:, a, :] + X[:, b, :])) for a, b in itertools.combinations(range(nv), 2)]
    wk = np.stack(wk, axis=1)                                  # (ncells, nk)
    wbar = wk @ Ws                                             # int I(w) / vol
    if cell_scale is not None:
        wbar = wbar * cell_scale
    rows, cols, kv, mv = [], [], [], []
    load = np.zeros(mesh.nv)
    for i in range(nv):
        np.add.at(load, c[:, i], vol * (wk @ Wl[:, i]))
        for j in range(nv):
            rows.append(c[:, i])
            cols.append(c[:, j])
            kv.append(vol * wbar * np.einsum("ck,ck->c", G[:, i, :], G[:, j, :]))
            mv.append(vol * (wk @ Wm[:, i, j]))
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    return (_assemble(rows, cols, np.concatenate(kv), mesh.nv), _assemble(rows, cols, np.concatenate(mv), mesh.nv),
            load)


CURVILINEAR = {
    # kind: (dim, weight degree, weight function of the mesh coordinates)
    "1d_cylindrical": (1, 1, lambda x: x[:, 0]),
    "1d_spherical": (1, 2, lambda x: x[:, 0] * x[:, 0]),
    "2d_cylindrical": (2, 1, lambda x: x[:, 0]),
    "2d_spherical": (2, 2, lambda x: x[:, 0] * x[:, 0] * np.sin(x[:, 1])),
    "3d_spherical": (3, 2, lambda x: x[:, 0] * x[:, 0] * np.sin(x[:, 1])),
}


def curvilinear_mesh(kind, r_inner, r_outer, n, z_length=None):
    """IntervalMesh(nr, r_inner, r_outer) :804,960 / RectangleMesh(Point(r_inner,0), Point(r_outer, z_length|pi))
    :1096,1223 / BoxMesh(Point(r_inner,0,0), Point(r_outer, pi, 2pi)) :1360-1364."""
    if kind.startswith("1d"):
        return interval_mesh(n[0], r_inner, r_outer)
    if kind == "2d_cylindrical":
        return rectangle_mesh(r_inner, 0.0, r_outer, z_length, n[0], n[1])
    if kind == "2d_spherical":
        return rectangle_mesh(r_inner, 0.0, r_outer, np.pi, n[0], n[1])
    return box_mesh((r_inner, 0.0, 0.0), (r_outer, np.pi, 2.0 * np.pi), n[0], n[1], n[2])


def curvilinear_coords(kind, X):
    """Output embedding of the dof coordinates (:918, 1040, 1167, 1298-1303, 1439-1444)."""
    out = np.zeros((X.shape[0], 3))
    if kind.startswith("1d"):
        out[:, 0] = X[:, 0]
    elif kind == "2d_cylindrical":
        out[:, 0], out[:, 2] = X[:, 0], X[:, 1]
    elif kind == "2d_spherical":
        out[:, 0] = X[:, 0] * np.sin(X[:, 1])
        out[:, 2] = X[:, 0] * np.cos(X[:, 1])
    else:
        out[:, 0] = X[:, 0] * np.sin(X[:, 1]) * np.cos(X[:, 2])
        out[:, 1] = X[:, 0] * np.sin(X[:, 1]) * np.sin(X[:, 2])
        out[:, 2] = X[:, 0] * np.cos(X[:, 1])
    return out


def solve_heat_curvilinear(kind: str, r_inner: float, r_outer: float, n: Sequence[int], diffusivity: float,
                           T_initial: float = 20.0, dt: float = 0.01, num_steps: int = 50, steady: bool = False,
                           source_type: str = "none", source_value: float = 0.0, T_inner: float = 100.0,
                           T_outer: float = 20.0, T_boundary: float = 20.0, z_length: float = 2.0) -> Field:
    """_solve_heat_{1d_cylindrical,1d_spherical,2d_cylindrical,2d_spherical,3d_spherical}_raw restated."""
    dim, degree, wfun = CURVILINEAR[kind]
    mesh = curvilinear_mesh(kind, r_inner, r_outer, n, z_length)
    Kw, Mw, mw = assemble_weighted(mesh, wfun, degree)
    if dim == 1:
        bcs = []
        if r_inner > 1e-10:
            bcs.append((dirichlet_dofs(mesh, lambda x, ob: ob & near(x[:, 0], r_inner)), T_inner))
        bcs.append((dirichlet_dofs(mesh, lambda x, ob: ob & near(x[:, 0], r_outer)), T_outer))
    else:
        bcs = [(dirichlet_dofs(mesh, lambda x, ob: ob), T_boundary)]
    bc_dofs, bc_vals = _merge_bcs(bcs, mesh.nv)
    f = float(source_value) if source_type == "constant" else 0.0
    kappa = float(diffusivity)
    snaps, times = [], []
    if steady:
        A, b = apply_bc_rowwise((kappa * Kw).tocsr(), f * mw, bc_dofs, bc_vals)
        snaps.append(lu_solve(A, b))
        times.append(0.0)
    else:
        u = np.full(mesh.nv, float(T_initial))       # every initial_type falls back to the constant (:893-896)
        u[bc_dofs] = bc_vals
        snaps.append(u.copy())
        times.append(0.0)
        A, _ = apply_bc_rowwise((Mw + (dt * kappa) * Kw).tocsr(), np.zeros(mesh.nv), bc_dofs, bc_vals)
        lu = _ScaledLU(A.tocsr())
        for step in range(num_steps):
            b = Mw @ u + (dt * f) * mw
            b[bc_dofs] = bc_vals
            u = lu.solve(b)
            snaps.append(u.copy())
            times.append((step + 1) * dt)
    vals = np.array(snaps)
    coords = curvilinear_coords(kind, mesh.coords)
    if dim == 1:                                      # the 1D tools sort by r (:872-874)
        order = np.argsort(mesh.coords[:, 0], kind="stable")
        coords, vals = coords[order], vals[:, order]
    return Field(coords=coords, values=vals, times=np.array(times), dim=dim, meta={"kind": kind})


def solve_heat_3d_special(Lx, Ly, Lz, n, diffusivity, T_boundary=0.0, T_initial=20.0, dt=0.01, num_steps=20,
                          steady=False, source_type="none", source_value=0.0, geometry_type="box",
                          cylinder_radius=None, T_left=None, T_right=None, T_side=None, core_radius=None,
                          core_diffusivity=None, initial_type="constant", initial_amplitude=1.0,
                          initial_wavenumber=1.0) -> Field:
    """The cylinder / composite-core branches of _solve_heat_3d_raw (:512-572, 576-605, 642-716) as they run in the
    reference's deployment, i.e. WITHOUT mshr (neither Dockerfile nor requirements.txt install it): the
    "cylinder" is BoxMesh(Point(0,-R,-R), Point(Lx,R,R), nx, int(ny*2R), int(nz*2R)) with every term weighted by
    Expression("sqrt(x[1]^2+x[2]^2)", degree=2); a composite core is a DG0 diffusivity equal to core_diffusivity on
    the cells SubDomain.mark selects for r < core_radius (all vertices and the midpoint inside)."""
    nx, ny, nz = n
    cyl = geometry_type == "cylinder" and cylinder_radius is not None
    if cyl:
        R = cylinder_radius
        mesh = box_mesh((0.0, -R, -R), (Lx, R, R), nx, int(ny * R * 2), int(nz * R * 2))
        wfun, degree = (lambda x: np.sqrt(x[:, 1] ** 2 + x[:, 2] ** 2)), 2
    else:
        mesh = box_mesh((0.0, 0.0, 0.0), (Lx, Ly, Lz), nx, ny, nz)
        wfun, degree = (lambda x: np.ones(x.shape[0])), 1
    kcell = None
    if core_radius is not None and core_diffusivity is not None:
        X = mesh.coords[mesh.cells]                                       # (nc, 4, 3)
        rv = np.sqrt(X[:, :, 1] ** 2 + X[:, :, 2] ** 2)
        mid = X.mean(axis=1)
        inside = (rv < core_radius).all(axis=1) & (np.sqrt(mid[:, 1] ** 2 + mid[:, 2] ** 2) < core_radius)
        kcell = np.where(inside, float(core_diffusivity), float(diffusivity))
    else:
        kcell = np.full(mesh.cells.shape[0], float(diffusivity))
    Kk, Mw, mw = assemble_weighted(mesh, wfun, degree, cell_scale=kcell)   # Kk already carries kappa
    directional = T_left is not None or T_right is not None or T_side is not None
    if directional:
        bcs = []
        if cyl:
            def side(x, ob):
                r = np.sqrt(x[:, 1] ** 2 + x[:, 2] ** 2)
                return ob & ~(near(x[:, 0], 0.0) | near(x[:, 0], Lx)) & near(r, cylinder_radius)
        else:
            def side(x, ob):
                return ob & ~(near(x[:, 0], 0.0) | near(x[:, 0], Lx))
        if T_left is not None:
            bcs.append((dirichlet_dofs(mesh, lambda x, ob: ob & near(x[:, 0], 0.0)), T_left))
        if T_right is not None:
            bcs.append((dirichlet_dofs(mesh, lambda x, ob: ob & near(x[:, 0], Lx)), T_right))
        if T_side is not None:
            bcs.append((dirichlet_dofs(mesh, side), T_side))
    else:
        bcs = [(dirichlet_dofs(mesh, lambda x, ob: ob), T_boundary)]
    bc_dofs, bc_vals = _merge_bcs(bcs, mesh.nv)
    f = float(source_value) if source_type == "constant" else 0.0
    snaps, times = [], []
    if steady:
        A, b = apply_bc_rowwise(Kk.tocsr(), f * mw, bc_dofs, bc_vals)
        snaps.append(lu_solve(A, b))
        times.append(0.0)
    else:
        if initial_type == "zero":
            u = np.zeros(mesh.nv)
        elif initial_type in ("cosine", "sine"):                    # unweighted project(), :674-685
            u = project_p2_expression(mesh, _initial_expression(3, initial_type, initial_amplitude,
                                                                initial_wavenumber))
        else:
            u = np.full(mesh.nv, float(T_initial))
        u[bc_dofs] = bc_vals
        snaps.append(u.copy())
        times.append(0.0)
        A, _ = apply_bc_rowwise((Mw + dt * Kk).tocsr(), np.zeros(mesh.nv), bc_dofs, bc_vals)
        lu = _ScaledLU(A.tocsr())
        for step in range(num_steps):
            b = Mw @ u + (dt * f) * mw
            b[bc_dofs] = bc_vals
            u = lu.solve(b)
            snaps.append(u.copy())
            times.append((step + 1) * dt)
    return Field(coords=mesh.coords.copy(), values=np.array(snaps), times=np.array(times), dim=3,
                 meta={"geometry_type": geometry_type})
