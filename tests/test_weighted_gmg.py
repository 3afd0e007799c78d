"""Galerkin multigrid for the weighted (curvilinear / cylinder / composite-core) heat operators.

CPU part: the NumPy model of the GPU hierarchy (build_galerkin below, on top of oracle.gmg_model) keeps the Kuhn
pattern, stays symmetric and converges in a bounded number of PCG iterations.  GPU part (pytest.mark.gpu):
precond="gmg" through the public functions against the oracle LU, the coarse operators against the model, the
iteration count against the model, and large grids against Jacobi-PCG on the same call."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import fem_oracle as fo
from oracle import gmg_model as gm

TOL = 1e-8


# ---------------------------------------------------------------- NumPy model of the GPU hierarchy (csrc/wmg.cu)
def build_galerkin(A, free, n, dim, dense_max=768):
    """Level 0 is the free-free block F A F of the assembled matrix A (natural vertex order, `free` = non-Dirichlet
    vertices, n = cells per axis); coarser levels are Fc P^T A P Fc with the Kuhn prolongation of oracle.gmg_model,
    while every axis halves evenly and the coarse grid keeps a free vertex.  lmax = Gershgorin bound of D^-1 A over the
    free rows; dense inverse of the (symmetrised) coarsest free block when it has <= dense_max free vertices.  The
    levels plug into oracle.gmg_model.vcycle / pcg."""
    n = list(n)
    free = np.asarray(free, dtype=bool)
    F = sp.diags(free.astype(float))
    Am = (F @ A @ F).tocsr()
    levels = []
    while True:
        lv = gm.Level()
        lv.n, lv.free, lv.Am = list(n), free, Am
        d = Am.diagonal()
        lv.dinv = np.where(free, 1.0 / np.where(free, d, 1.0), 0.0)
        lv.lmax = float(np.max(np.asarray(abs(Am).sum(axis=1)).ravel()[free] / d[free]))
        levels.append(lv)
        if not all(k % 2 == 0 and k >= 2 for k in n):
            break
        nc = [k // 2 for k in n]
        nnf = [k + 1 for k in n]
        X = np.indices([k + 1 for k in nc][::-1]).reshape(dim, -1)[::-1]     # coarse (x, y, z), x fastest
        fine_of_coarse = sum(2 * X[q] * int(np.prod(nnf[:q])) for q in range(dim))
        free_c = free[fine_of_coarse]
        if not free_c.any():
            break
        lv.P = gm.prolongation(n + [0] * (3 - dim))
        Fc = sp.diags(free_c.astype(float))
        Am = (Fc @ (lv.P.T @ Am @ lv.P) @ Fc).tocsr()
        free, n = free_c, nc
    lc = levels[-1]
    idx = np.nonzero(lc.free)[0]
    lc.dense = None
    if len(levels) > 1 and idx.size <= dense_max:
        B = lc.Am[idx][:, idx].toarray()
        lc.idx = idx
        lc.dense = np.linalg.inv(0.5 * (B + B.T))
    return levels


# ---------------------------------------------------------------- systems (steady operators, natural vertex order)
def curvi_system(kind, n, r_inner, r_outer=1.0, z_length=2.0, kappa=1.0):
    dim, degree, wfun = fo.CURVILINEAR[kind]
    mesh = fo.curvilinear_mesh(kind, r_inner, r_outer, n, z_length)
    Kw, _, mw = fo.assemble_weighted(mesh, wfun, degree)
    if dim == 1:
        dofs = fo.dirichlet_dofs(mesh, lambda x, ob: ob & fo.near(x[:, 0], r_outer))
        if r_inner > 1e-10:
            dofs = np.union1d(dofs, fo.dirichlet_dofs(mesh, lambda x, ob: ob & fo.near(x[:, 0], r_inner)))
    else:
        dofs = fo.dirichlet_dofs(mesh, lambda x, ob: ob)
    free = np.ones(mesh.nv, dtype=bool)
    free[dofs] = False
    return (kappa * Kw).tocsr(), free, mw, dim


def cylinder_core_system(n, R=0.5, core_radius=0.25, kappa=1.0, core_factor=25.0):
    """BoxMesh (0,-R,-R)-(1,R,R), weight sqrt(y^2+z^2) (degree 2), DG0 core diffusivity, all faces Dirichlet."""
    mesh = fo.box_mesh((0.0, -R, -R), (1.0, R, R), *n)
    X = mesh.coords[mesh.cells]
    rv = np.sqrt(X[:, :, 1] ** 2 + X[:, :, 2] ** 2)
    mid = X.mean(axis=1)
    inside = (rv < core_radius).all(axis=1) & (np.sqrt(mid[:, 1] ** 2 + mid[:, 2] ** 2) < core_radius)
    kcell = np.where(inside, core_factor * kappa, kappa)
    K, _, mw = fo.assemble_weighted(mesh, lambda x: np.sqrt(x[:, 1] ** 2 + x[:, 2] ** 2), 2, cell_scale=kcell)
    free = np.ones(mesh.nv, dtype=bool)
    free[fo.dirichlet_dofs(mesh, lambda x, ob: ob)] = False
    return K.tocsr(), free, mw, 3


def kuhn_offsets(dim):
    off = {(0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, 0, 1), (0, 1, 1), (1, 1, 1)}
    off |= {tuple(-v for v in o) for o in off}
    return {o for o in off if all(o[q] == 0 for q in range(dim, 3))}


def vertex_xyz(n, dim):
    nn = [k + 1 for k in n]
    return np.indices(nn[::-1]).reshape(dim, -1)[::-1].T          # (nverts, dim), x fastest


def model_pcg_iters(levels, b):
    _, hist = gm.pcg(levels, b, rtol=1e-10, max_iters=400)
    assert hist[-1] <= 1e-10
    return len(hist)


# ---------------------------------------------------------------- CPU: the model hierarchy
@pytest.mark.parametrize("name,system,n", [
    ("2d_spherical", lambda n: curvi_system("2d_spherical", n, 0.0), [32, 32]),
    ("3d_spherical", lambda n: curvi_system("3d_spherical", n, 0.2), [16, 16, 16]),
    ("cylinder_core", cylinder_core_system, [16, 16, 16]),
])
def test_galerkin_levels_keep_kuhn_pattern_and_symmetry(name, system, n):
    A, free, _, dim = system(n)
    levels = build_galerkin(A, free, n, dim)
    assert len(levels) >= 3
    allowed = kuhn_offsets(dim)
    for lv in levels[1:]:
        C = lv.Am.tocoo()
        scale = abs(C.data).max()
        big = abs(C.data) > 1e-14 * scale
        xyz = vertex_xyz(lv.n, dim)
        d = xyz[C.col[big]] - xyz[C.row[big]]
        d3 = np.zeros((d.shape[0], 3), dtype=int)
        d3[:, :dim] = d
        assert {tuple(v) for v in d3} <= allowed, name
        assert abs(lv.Am - lv.Am.T).max() <= 1e-14 * scale, name
        assert not (abs(lv.Am)[~lv.free].sum() or abs(lv.Am)[:, ~lv.free].sum())   # free-free block only


@pytest.mark.parametrize("name,system,n,bound", [
    ("2d_cylindrical", lambda n: curvi_system("2d_cylindrical", n, 0.0), [256, 256], 16),
    ("2d_spherical", lambda n: curvi_system("2d_spherical", n, 0.0), [256, 256], 30),
    ("cylinder_core", cylinder_core_system, [32, 32, 32], 16),
    ("3d_spherical", lambda n: curvi_system("3d_spherical", n, 0.2), [32, 32, 32], 42),
])
def test_galerkin_model_pcg_iteration_bounds(name, system, n, bound):
    A, free, _, dim = system(n)
    levels = build_galerkin(A, free, n, dim)
    b = np.random.default_rng(0).standard_normal(A.shape[0])
    assert model_pcg_iters(levels, b) <= bound, name


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def P():
    import pde_solver_b200 as p
    return p


def _gmg_stats_ok(P):
    st = P.last_stats()
    assert st["converged"] == 1 and st["levels"] >= 2 and st["true_relres"] <= 1e-9, st
    return st


CURVI = [
    ("1d_cylindrical", [64], dict(r_inner=0.1, r_outer=1.0, T_inner=100.0, T_outer=20.0)),
    ("1d_cylindrical", [64], dict(r_inner=0.0, r_outer=1.0, T_inner=100.0, T_outer=20.0)),
    ("1d_spherical", [64], dict(r_inner=0.1, r_outer=1.0, T_inner=100.0, T_outer=20.0)),
    ("2d_cylindrical", [32, 32], dict(r_inner=0.1, r_outer=1.0, z_length=2.0, T_boundary=35.0)),
    ("2d_spherical", [32, 32], dict(r_inner=0.1, r_outer=1.0, T_boundary=35.0)),
    ("3d_spherical", [16, 8, 16], dict(r_inner=0.2, r_outer=1.0, T_boundary=35.0)),
]
NAMES = {"1d_cylindrical": ["nr"], "1d_spherical": ["nr"], "2d_cylindrical": ["nr", "nz"],
         "2d_spherical": ["nr", "ntheta"], "3d_spherical": ["nr", "ntheta", "nphi"]}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,kw", CURVI)
@pytest.mark.parametrize("steady", [False, True])
def test_curvilinear_gmg_matches_oracle(P, kind, n, kw, steady):
    common = dict(diffusivity=0.8, T_initial=20.0, dt=0.02, num_steps=4, steady=steady, source_type="constant",
                  source_value=40.0)
    ref = fo.solve_heat_curvilinear(kind, kw["r_inner"], kw["r_outer"], n,
                                    **{k: v for k, v in kw.items() if k not in ("r_inner", "r_outer")}, **common)
    fn = getattr(P, f"_solve_heat_{kind}_raw")
    f = fn(**kw, **dict(zip(NAMES[kind], n)), **common, precond="gmg", as_arrays=True)
    assert f.values.shape == ref.values.shape
    for k in range(ref.values.shape[0]):
        assert fo.rel_l2(f.values[k], ref.values[k]) <= TOL, (k, fo.rel_l2(f.values[k], ref.values[k]))
    _gmg_stats_ok(P)


CYL_CORE = [
    dict(geometry_type="cylinder", T_boundary=1.0, T_initial=5.0, source_type="constant", source_value=3.0),
    dict(geometry_type="cylinder", T_left=10.0, T_right=2.0, T_side=50.0, T_initial=4.0),
    dict(geometry_type="cylinder", T_side=7.0, T_initial=4.0, source_type="constant", source_value=1.0),
    dict(core_radius=0.3, core_diffusivity=25.0, T_boundary=0.0, T_initial=3.0),
    dict(core_radius=0.3, core_diffusivity=25.0, T_left=1.0, T_side=2.0, T_initial=3.0),
    dict(geometry_type="cylinder", core_radius=0.15, core_diffusivity=8.0, steady=True, T_boundary=2.0,
         source_type="constant", source_value=5.0),
    dict(core_radius=0.3, core_diffusivity=4.0, T_boundary=0.5, initial_type="cosine", initial_amplitude=2.0,
         initial_wavenumber=3.0),
    dict(geometry_type="cylinder", T_boundary=0.0, initial_type="sine", initial_amplitude=1.5, initial_wavenumber=4.0),
    dict(geometry_type="cylinder", T_boundary=0.0, initial_type="zero", source_type="constant", source_value=2.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CYL_CORE)
def test_cylinder_and_composite_core_gmg_matches_oracle(P, case):
    # the cases of the Jacobi parity test on even grids: box 8x16x16, cylinder radius 0.5 -> BoxMesh 8x16x16
    Lx, Ly, Lz, n, kappa = 1.0, 0.5, 0.5, [8, 16, 16], 0.8
    kw = dict(dt=0.02, num_steps=3)
    kw.update(case)
    if case.get("geometry_type") == "cylinder":
        kw["cylinder_radius"] = 0.5
    ref = fo.solve_heat_3d_special(Lx, Ly, Lz, n, kappa, **kw)
    args = dict(T_boundary=0.0, T_initial=0.0, steady=False)
    args.update(kw)
    f = P._solve_heat_3d_raw(Lx, Ly, Lz, n[0], n[1], n[2], kappa, args.pop("T_boundary"), args.pop("T_initial"),
                             args.pop("dt"), args.pop("num_steps"), precond="gmg", as_arrays=True, **args)
    v = np.asarray(f.values)
    assert v.shape == ref.values.shape
    for a, b in zip(v, ref.values):
        assert np.linalg.norm(a - b) <= TOL * max(np.linalg.norm(b), 1e-300)
    _gmg_stats_ok(P)


def _wheat_params(P, dim, n, lo, hi, rpow=0, wsin=0, degree=1, kind=0, core=None, kappa=1.0, faces=None):
    L = P._lib
    p = L.WheatParams()
    p.dim = dim
    p.n = L.i3(n)
    p.lo = L.d3(lo, 0.0)
    p.hi = L.d3(hi, 1.0)
    p.weight_rpow, p.weight_sin_axis1, p.weight_degree, p.weight_kind = rpow, wsin, degree, kind
    if core is not None:
        p.has_core, p.core_radius, p.core_diffusivity = 1, core[0], core[1]
    p.steady = 1
    p.diffusivity = kappa
    p.bc = L.make_bc(faces if faces is not None else {f: 0.0 for f in range(2 * dim)})
    return p


def _level_matrix(P, p, level, dim):
    import ctypes as C
    L = P._lib
    ctx = L.default_context()
    n_out = (C.c_int32 * 3)()
    L.check(L.lib().pde_wheat_level_coefs(ctx.handle, C.byref(p), level, n_out, None))
    n = [n_out[q] for q in range(dim)]
    nv = int(np.prod([k + 1 for k in n]))
    nk = {1: 3, 2: 7, 3: 15}[dim]
    coef = np.empty((nk, nv))
    L.check(L.lib().pde_wheat_level_coefs(ctx.handle, C.byref(p), level, n_out, L.ptr(coef)))
    # offsets in internal axes (2-D: x, z = user x, y)
    full = [(0, 0, 0), (1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1), (1, 1, 0), (-1, -1, 0),
            (1, 0, 1), (-1, 0, -1), (0, 1, 1), (0, -1, -1), (1, 1, 1), (-1, -1, -1)]
    if dim == 1:
        offs = [o[:1] for o in full[:3]]
    elif dim == 2:
        offs = [(o[0], o[2]) for o in full if o[1] == 0]
    else:
        offs = full
    xyz = vertex_xyz(n, dim)
    nn = np.array([k + 1 for k in n])
    rows, cols, vals = [], [], []
    for k, o in enumerate(offs):
        t = xyz + np.array(o)
        ok = np.all((t >= 0) & (t < nn), axis=1)
        j = sum(t[:, q] * int(np.prod(nn[:q])) for q in range(dim))
        rows.append(np.nonzero(ok)[0])
        cols.append(j[ok])
        vals.append(coef[k][ok])
        assert not np.any(coef[k][~ok]), "entry towards a vertex outside the grid"
    return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(nv, nv)), n


COARSE_CASES = [
    ("2d_spherical", [32, 32]),
    ("3d_spherical", [16, 8, 16]),
    ("cylinder_core", [8, 16, 16]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", COARSE_CASES)
def test_level_coefs_match_galerkin_model(P, name, n):
    if name == "cylinder_core":
        A, free, _, dim = cylinder_core_system(n)
        p = _wheat_params(P, 3, n, [0.0, -0.5, -0.5], [1.0, 0.5, 0.5], degree=2, kind=1, core=(0.25, 25.0))
    else:
        r_inner = 0.2 if name == "3d_spherical" else 0.1
        A, free, _, dim = curvi_system(name, n, r_inner)
        hi = [1.0, np.pi, 2 * np.pi][:dim]
        p = _wheat_params(P, dim, n, [r_inner, 0.0, 0.0][:dim], hi, rpow=2, wsin=1, degree=2)
    levels = build_galerkin(A, free, n, dim)
    scale = abs(A).max()
    for level in (0, 1, 2):
        G, nl = _level_matrix(P, p, level, dim)
        assert nl == levels[level].n
        err = abs(G - levels[level].Am).max()
        assert err <= 1e-13 * scale, (level, err / scale)
    import ctypes as C
    n_out = (C.c_int32 * 3)()
    assert P._lib.lib().pde_wheat_level_coefs(P._lib.default_context().handle, C.byref(p), len(levels), n_out,
                                              None) != 0


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", [("2d_spherical", [64, 64]), ("3d_spherical", [16, 16, 16]),
                                    ("cylinder_core", [32, 32, 32])])
def test_vcycle_matches_galerkin_model(P, name, n):
    """pde_wheat_vcycle (the V-cycle of the GMG-PCG) against oracle.gmg_model.vcycle on the Galerkin model, vector by
    vector: a wrong V-cycle kernel slows the solve down without changing its solution."""
    if name == "cylinder_core":
        A, free, _, dim = cylinder_core_system(n)
        p = _wheat_params(P, 3, n, [0.0, -0.5, -0.5], [1.0, 0.5, 0.5], degree=2, kind=1, core=(0.25, 25.0))
    else:
        r_inner = 0.2 if name == "3d_spherical" else 0.1
        A, free, _, dim = curvi_system(name, n, r_inner)
        hi = [1.0, np.pi, 2 * np.pi][:dim]
        p = _wheat_params(P, dim, n, [r_inner, 0.0, 0.0][:dim], hi, rpow=2, wsin=1, degree=2)
    levels = build_galerkin(A, free, n, dim)
    b = np.random.default_rng(4).standard_normal(A.shape[0]) * free
    z1, z3, bz, info = P._lib.wheat_vcycle(P._lib.default_context(), p, b, ncycles=3)
    assert info["levels"] == len(levels)
    assert info["n_dense"] == (levels[-1].idx.size if levels[-1].dense is not None else 0)
    for l, lv in enumerate(levels):
        assert info["n"][l][:dim] == lv.n
        assert abs(info["lmax"][l] - lv.lmax) <= 1e-13 * lv.lmax, (l, info["lmax"][l], lv.lmax)
    ref = gm.vcycle(levels, b)
    ratio = np.abs(z1 - ref).max() / np.abs(ref).max()
    print(f"[wvcycle] {name} {n}: max|z-z_model|/max|z_model| = {ratio:.2e}")
    assert ratio <= 1e-11, ratio
    assert not z1[~free].any()
    assert np.array_equal(z3, z1)
    assert abs(bz - b @ z1) <= 1e-12 * np.abs(b * z1).sum()
    assert info["paths"] == [0] * len(levels) and info["graph"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["2d_spherical_64", "cylinder_core_32"])
def test_gmg_iterations_match_model(P, name):
    f_src, Tb = 40.0, 35.0
    if name == "2d_spherical_64":
        n = [64, 64]
        A, free, mw, dim = curvi_system("2d_spherical", n, 0.0)
        P._solve_heat_2d_spherical_raw(0.0, 1.0, 64, 64, 1.0, Tb, 0.0, 0.01, 1, steady=True, source_type="constant",
                                       source_value=f_src, precond="gmg", as_arrays=True)
    else:
        n = [32, 32, 32]
        A, free, mw, dim = cylinder_core_system(n)
        P._solve_heat_3d_raw(1.0, 1.0, 1.0, 32, 32, 32, 1.0, Tb, 0.0, 0.01, 1, steady=True, source_type="constant",
                             source_value=f_src, geometry_type="cylinder", cylinder_radius=0.5, core_radius=0.25,
                             core_diffusivity=25.0, precond="gmg", as_arrays=True)
    st = _gmg_stats_ok(P)
    u_lift = np.where(free, 0.0, Tb)
    b = np.where(free, f_src * mw - A @ u_lift, 0.0)
    levels = build_galerkin(A, free, n, dim)
    assert st["levels"] == len(levels)
    it = model_pcg_iters(levels, b)
    assert abs(st["iters_total"] - it) <= 2, (st["iters_total"], it)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["2d_spherical_2048", "core_box_256"])
def test_gmg_scales_and_agrees_with_jacobi(P, name):
    def solve(precond, rtol):
        if name == "2d_spherical_2048":
            f = P._solve_heat_2d_spherical_raw(0.0, 1.0, 2048, 2048, 1.0, 35.0, 0.0, 0.01, 1, steady=True,
                                               source_type="constant", source_value=40.0, rtol=rtol,
                                               precond=precond, as_arrays=True)
        else:
            f = P._solve_heat_3d_raw(1.0, 1.0, 1.0, 256, 256, 256, 1.0, 0.0, 0.0, 0.01, 1, steady=True,
                                     source_type="constant", source_value=40.0, core_radius=0.3,
                                     core_diffusivity=25.0, rtol=rtol, precond=precond, as_arrays=True)
        return np.asarray(f.values[-1]), P.last_stats()

    _, st = solve("gmg", 1e-10)
    assert st["levels"] >= 6 and st["iters_total"] <= 40 and st["true_relres"] <= 1e-9, st
    # the two preconditioners agree to 1e-8 once both solves are tight: at rtol 1e-10 the algebraic error of a
    # 4 M-dof Laplacian-like system (condition ~ h^-2) can exceed 1e-8 on its own
    vg, _ = solve("gmg", 1e-12)
    vj, sj = solve("jacobi", 1e-12)
    assert sj["levels"] == 1
    assert fo.rel_l2(vg, vj) <= TOL


@pytest.mark.gpu
def test_odd_grid_falls_back_to_jacobi(P):
    P._solve_heat_2d_spherical_raw(0.1, 1.0, 15, 16, 1.0, 35.0, 0.0, 0.01, 1, steady=True, source_type="constant",
                                   source_value=40.0, precond="gmg", as_arrays=True)
    st = P.last_stats()
    assert st["levels"] == 1 and st["converged"] == 1
