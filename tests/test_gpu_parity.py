"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.

Bars (BASELINE.json north_star): mesh / dof maps / boundary sets bit-exact; nodal solutions within
1e-8 relative L2 of the direct-LU oracle at solver rtol 1e-10."""
import numpy as np
import pytest

from oracle import fem_oracle as fo

pytestmark = pytest.mark.gpu

TOL = 1e-8  # relative L2, FP64, north_star


@pytest.fixture(scope="module")
def P():
    import pde_solver_b200 as p
    return p


@pytest.fixture(scope="module")
def ctx(P):
    return P._lib.default_context()


# ---------------------------------------------------------------- meshes / dof maps / boundary sets
@pytest.mark.parametrize("dim,n,L", [(1, [100], [2.0]), (1, [7], [0.3]), (2, [5, 3], [1.0, 0.6]),
                                     (2, [10, 10], [0.2, 0.2]), (3, [4, 3, 2], [1.0, 0.2, 0.2]),
                                     (3, [10, 7, 5], [0.3, 0.2, 0.7]), (3, [1, 1, 1], [1, 1, 1])])
def test_mesh_bit_exact(P, dim, n, L):
    m = fo.make_mesh(dim, L, n)
    assert np.array_equal(P.mesh.coordinates(dim, n, L), m.coords)          # FP64 bit-exact
    assert np.array_equal(P.mesh.cells(dim, n, ordered=False), m.cells_raw)
    assert np.array_equal(P.mesh.cells(dim, n, ordered=True), m.cells)
    assert np.array_equal(P.mesh.cell_dofs(dim, n, 1), fo.cell_dofs_scalar(m))
    if dim > 1:
        for layout in ("blocked", "interleaved"):
            assert np.array_equal(P.mesh.cell_dofs(dim, n, dim, layout), fo.cell_dofs_vector(m, dim, layout))


@pytest.mark.parametrize("dim,n", [(1, [9]), (2, [5, 4]), (3, [4, 3, 2]), (3, [2, 3, 2]), (3, [3, 1, 1])])
def test_boundary_sets_bit_exact(P, dim, n):
    L = [1.0, 0.7, 0.4][:dim]
    m = fo.make_mesh(dim, L, n)
    cases = [dict(T_boundary=3.0)] if dim > 1 else [dict(T_left=20.0, T_right=1.0)]
    if dim == 3:
        cases += [dict(T_left=1.0), dict(T_side=2.0), dict(T_left=1.0, T_right=2.0, T_side=3.0),
                  dict(T_right=4.0, T_side=5.0)]
    for kw in cases:
        dofs, vals = fo._merge_bcs(fo.heat_bcs(m, L, **kw), m.nv)
        mask, v = P.mesh.dirichlet(dim, n, P.mesh.heat_bc(dim, **kw))
        assert np.array_equal(np.nonzero(mask)[0], dofs), kw
        assert np.array_equal(v[dofs], vals), kw
    # elasticity clamp: near(x[0], 0) plane
    clamp = fo.dirichlet_dofs(m, lambda x, ob: fo.near(x[:, 0], 0.0))
    mask, _ = P.mesh.dirichlet(dim, n, P._lib.make_bc({0: 0.0}))
    assert np.array_equal(np.nonzero(mask)[0], clamp)


# ---------------------------------------------------------------- operator application
def _oracle_matrix(kind, dim, n, L, alpha, beta, lam, mu):
    m = fo.make_mesh(dim, L, n)
    if kind == "elasticity":
        A = fo.assemble_elasticity(m, lam, mu)      # interleaved dofs
        nv = m.nv
        perm = (np.arange(dim)[:, None] + dim * np.arange(nv)[None, :]).ravel()   # blocked -> interleaved
        return m, A[perm][:, perm].tocsr()
    K, M = fo.assemble_stiffness_mass(m)
    return m, (alpha * M + beta * K).tocsr()


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("kind,dim,n", [("heat", 1, [33]), ("heat", 2, [17, 9]), ("heat", 3, [9, 6, 7]),
                                        ("heat", 3, [40, 12, 10]), ("mass", 3, [5, 5, 5]),
                                        ("stiffness", 2, [8, 8]), ("elasticity", 2, [9, 7]),
                                        ("elasticity", 3, [6, 5, 4]), ("elasticity", 3, [36, 6, 5]),
                                        ("heat", 3, [1, 1, 1]), ("elasticity", 3, [2, 1, 3]),
                                        # sizes that take the TMA plane-sweep kernel (several x/y tiles, z chunks)
                                        ("heat", 3, [70, 33, 40]), ("mass", 3, [64, 20, 9]),
                                        ("heat", 3, [400, 10, 8]), ("elasticity", 3, [66, 20, 12]),
                                        ("elasticity", 3, [200, 9, 36]),
                                        # 2-D sizes that take the register-marching kernel when every face is Dirichlet
                                        ("heat", 2, [300, 70]), ("mass", 2, [129, 200]), ("stiffness", 2, [256, 9])])
def test_operator_apply_matches_oracle(P, ctx, kind, dim, n, variant):
    L = [1.0, 0.6, 0.35][:dim]
    alpha, beta = (1.0, 0.013) if kind == "heat" else ((1.0, 0.0) if kind == "mass" else (0.0, 1.0))
    lam, mu = fo.lame(210e9, 0.3, 3)
    m, A = _oracle_matrix(kind, dim, n, L, alpha, beta, lam, mu)
    nc = dim if kind == "elasticity" else 1
    rng = np.random.default_rng(0)
    x = rng.standard_normal((nc, m.nv))
    for bc, dofs in ((None, np.array([], dtype=int)),
                     (P._lib.make_bc({0: 0.0}), fo.dirichlet_dofs(m, lambda xx, ob: fo.near(xx[:, 0], 0.0))),
                     (P._lib.make_bc({f: 0.0 for f in range(2 * dim)}),
                      fo.dirichlet_dofs(m, lambda xx, ob: np.ones(xx.shape[0], bool)))):
        p = P._lib.op_params(kind, dim, n, L, alpha, beta, lam, mu, bc=bc, variant=variant)
        y = P._lib.op_apply(ctx, p, x)
        ref = (A @ x.ravel()).reshape(nc, m.nv)
        ref[:, dofs] = 0.0                                  # Dirichlet rows are masked
        scale = np.abs(A).max() * np.abs(x).max()
        assert np.abs(y - ref).max() <= 1e-13 * scale * 30
        # the constant right-hand-side term of the same launch (heat source f m, body force): g (.) m - A x
        g = np.array([0.7, -1.3, 2.1])
        yl = P._lib.op_load(ctx, p, g, x)
        refl = g[:nc, None] * fo.lumped_load(m)[None, :] - (A @ x.ravel()).reshape(nc, m.nv)
        refl[:, dofs] = 0.0
        ratio = np.abs(yl - refl).max() / max(scale, np.abs(refl).max())
        # with x = 0 the load term stands alone (next to A x it is ~1e-12 of the elasticity operator's scale)
        m0 = np.where(np.isin(np.arange(m.nv), dofs), 0.0, fo.lumped_load(m))
        y0 = P._lib.op_load(ctx, p, g, np.zeros_like(x))
        ratio0 = (np.abs(y0 - g[:nc, None] * m0[None, :]).max()
                  / max(np.abs(g).max() * m0.max(), np.finfo(float).tiny))
        print(f"[op_load] {kind} {dim}d {n} variant {variant} dirichlet {len(dofs)}: ratio {ratio:.2e}, "
              f"x = 0 {ratio0:.2e}")
        assert ratio <= 1e-13 * 30 and ratio0 <= 1e-13 * 30


@pytest.mark.parametrize("kind,n", [("elasticity", [66, 20, 12]), ("elasticity", [40, 9, 37]), ("heat", [70, 33, 40])])
def test_fused_first_two_sweeps_match_oracle(P, ctx, kind, n):
    """Mode 5: x1 = s0 D^-1 b, y = (1 + c1) x1 + c2 D^-1 (b - A x1) in one pass.  Heat: uniform-diagonal operators only
    (every face Dirichlet).  Elasticity: any face set - k_elast3d with column-scaled coefficients inside, the two-layer
    face kernel with the class diagonal of every neighbour on and next to the natural faces."""
    dim, L = 3, [1.0, 0.6, 0.35]
    alpha, beta = (1.0, 0.013) if kind == "heat" else (1.0, 0.0)
    lam, mu = fo.lame(210e9, 0.3, 3)
    m, A = _oracle_matrix(kind, dim, n, L, alpha, beta, lam, mu)
    nc = dim if kind == "elasticity" else 1
    rng = np.random.default_rng(2)
    b = rng.standard_normal((nc, m.nv))
    dinv = 1.0 / A.diagonal().reshape(nc, m.nv)
    c1, s0 = 0.37, 0.8 / np.abs(A).sum(axis=1).max() * A.diagonal().max()
    cases = [{f: 0.0 for f in range(6)}] if kind == "heat" else [{}, {0: 0.0}, {0: 0.0, 3: 0.0, 4: 0.0}, {f: 0.0 for f in range(6)}]
    for faces in cases:
        on = [f in faces for f in range(6)]

        def pred(xx, ob):
            sel = np.zeros(xx.shape[0], bool)
            for ax in range(3):
                if on[2 * ax]:
                    sel |= fo.near(xx[:, ax], 0.0)
                if on[2 * ax + 1]:
                    sel |= fo.near(xx[:, ax], L[ax])
            return sel
        dofs = fo.dirichlet_dofs(m, pred) if faces else np.array([], dtype=int)
        free = np.ones((nc, m.nv))
        free[:, dofs] = 0.0
        bm = free * b                                      # a smoother right-hand side vanishes on the Dirichlet rows
        x1 = s0 * dinv * bm
        ref = free * ((1.0 + c1) * x1 + s0 * dinv * (bm - (A @ x1.ravel()).reshape(nc, m.nv)))
        p = P._lib.op_params(kind, dim, n, L, alpha, beta, lam, mu, bc=P._lib.make_bc(faces))
        y, _ = P._lib.op_sweep(ctx, p, 5, bm, bm, None, c1, s0)
        assert np.abs(y - ref).max() <= 3e-12 * max(np.abs(ref).max(), 1.0), faces


@pytest.mark.parametrize("kind,n", [("elasticity", [66, 20, 12]), ("elasticity", [40, 9, 37]), ("elasticity", [200, 9, 36]),
                                    ("heat", [70, 33, 40]), ("mass", [64, 20, 9])])
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_sweep_modes_match_oracle_and_generic_kernel(P, ctx, kind, n, mode):
    """Every mode of the specialised plane-sweep kernels (apply, residual, Chebyshev restart / with the previous
    iterate written in place / from a zero previous iterate) against the oracle matrix and the generic table kernel."""
    dim, L = 3, [1.0, 0.6, 0.35]
    alpha, beta = (1.0, 0.013) if kind == "heat" else (1.0, 0.0)
    lam, mu = fo.lame(210e9, 0.3, 3)
    m, A = _oracle_matrix(kind, dim, n, L, alpha, beta, lam, mu)
    nc = dim if kind == "elasticity" else 1
    rng = np.random.default_rng(1)
    x, b, xp = (rng.standard_normal((nc, m.nv)) for _ in range(3))
    dinv = 1.0 / A.diagonal().reshape(nc, m.nv)
    c1, c2 = 0.37, 0.8 / np.abs(A).sum(axis=1).max() * A.diagonal().max()
    for faces in ({}, {0: 0.0}, {0: 0.0, 3: 0.0, 4: 0.0}, {f: 0.0 for f in range(6)}):
        on = [f in faces for f in range(6)]

        def pred(xx, ob):
            sel = np.zeros(xx.shape[0], bool)
            for ax in range(3):
                if on[2 * ax]:
                    sel |= fo.near(xx[:, ax], 0.0)
                if on[2 * ax + 1]:
                    sel |= fo.near(xx[:, ax], L[ax])
            return sel
        dofs = fo.dirichlet_dofs(m, pred) if faces else np.array([], dtype=int)
        free = np.ones((nc, m.nv))
        free[:, dofs] = 0.0
        Ax = (A @ x.ravel()).reshape(nc, m.nv)
        if mode == 0:
            ref = free * Ax
        elif mode == 1:
            ref = free * (b - Ax)
        else:
            d = {2: 0.0, 3: x - xp, 4: x}[mode]
            ref = x + free * ((0.0 if mode == 2 else c1) * d + c2 * dinv * (b - Ax))
        out = {}
        for variant in (0, 1):
            p = P._lib.op_params(kind, dim, n, L, alpha, beta, lam, mu, bc=P._lib.make_bc(faces), variant=variant)
            out[variant], dots = P._lib.op_sweep(ctx, p, mode, x, b, xp, c1, c2)
            scale = max(np.abs(A).max() * np.abs(x).max(), np.abs(ref).max())
            assert np.abs(out[variant] - ref).max() <= 3e-12 * scale, (faces, variant)
            want = (x * ref).sum() if mode < 2 else (free * b * ref).sum()
            assert abs(dots[0] - want) <= 1e-9 * (np.abs(x * ref).sum() + np.abs(b * ref).sum()), (faces, variant)
        assert np.abs(out[0] - out[1]).max() <= 3e-12 * scale


# ---------------------------------------------------------------- heat solves vs oracle LU
def _check_heat(P, dim, L, n, okw, gkw, precond):
    ref = fo.solve_heat(dim, L, n, **okw)
    fn = {1: P._solve_heat_1d_raw, 2: P._solve_heat_2d_raw, 3: P._solve_heat_3d_raw}[dim]
    f = fn(*gkw["args"], **gkw["kw"], precond=precond, as_arrays=True)
    assert f.values.shape == ref.values.shape
    assert np.array_equal(np.asarray(f.coords), ref.coords)
    assert np.allclose(f.times, ref.times, rtol=0, atol=1e-15)
    for k in range(ref.values.shape[0]):
        assert fo.rel_l2(f.values[k], ref.values[k]) <= TOL, (k, fo.rel_l2(f.values[k], ref.values[k]))
    st = P.last_stats()
    assert st["converged"] == 1
    assert st["true_relres"] <= 1e-9, st      # recomputed b - A u of the last step, not the PCG recurrence
    return f, st


@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
def test_heat_1d_config1(P, precond):
    # BASELINE config 1: rod L=2, 100 cells, 20 / 0 Dirichlet, backward Euler (dispatcher: dt .01, 200 steps)
    okw = dict(diffusivity=1.0, T_initial=0.0, dt=0.01, num_steps=200, T_left=20.0, T_right=0.0)
    _check_heat(P, 1, [2.0], [100], okw,
                dict(args=(2.0, 100, 1.0, 20.0, 0.0, 0.0, 0.01, 200), kw={}), precond)


@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
def test_heat_2d(P, precond):
    okw = dict(diffusivity=1.0, T_initial=20.0, dt=0.01, num_steps=10, T_boundary=0.0)
    _check_heat(P, 2, [1.0, 1.0], [64, 64], okw,
                dict(args=(1.0, 1.0, 64, 64, 1.0, 0.0, 20.0, 0.01, 10), kw={}), precond)
    okw = dict(diffusivity=0.5, T_initial=5.0, dt=0.02, num_steps=4, T_boundary=7.0, source_type="constant",
               source_value=30.0)
    _check_heat(P, 2, [1.0, 0.5], [30, 18], okw,
                dict(args=(1.0, 0.5, 30, 18, 0.5, 7.0, 5.0, 0.02, 4),
                     kw=dict(source_type="constant", source_value=30.0)), precond)


@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
def test_heat_2d_marching_kernel_sizes(P, precond):
    """Grids wide enough for the register-marching 2-D sweep (k_sweep2d: >= 128 nodes across, all faces Dirichlet),
    ragged against its 256-column blocks and 64-row chunks; with a source, non-zero boundary value and a steady solve."""
    okw = dict(diffusivity=0.7, T_initial=3.0, dt=0.02, num_steps=4, T_boundary=2.0, source_type="constant",
               source_value=9.0)
    _check_heat(P, 2, [1.0, 0.4], [300, 70], okw,
                dict(args=(1.0, 0.4, 300, 70, 0.7, 2.0, 3.0, 0.02, 4),
                     kw=dict(source_type="constant", source_value=9.0)), precond)
    okw = dict(diffusivity=1.3, T_initial=0.0, dt=0.01, num_steps=1, T_boundary=1.0, steady=True,
               source_type="constant", source_value=5.0)
    _check_heat(P, 2, [0.5, 1.0], [128, 96], okw,
                dict(args=(0.5, 1.0, 128, 96, 1.3, 1.0, 0.0, 0.01, 1),
                     kw=dict(steady=True, source_type="constant", source_value=5.0)), precond)


@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
def test_heat_3d(P, precond):
    okw = dict(diffusivity=1.0, T_initial=20.0, dt=0.01, num_steps=5, T_boundary=0.0)
    _, st = _check_heat(P, 3, [1, 1, 1], [32, 32, 32], okw,
                        dict(args=(1, 1, 1, 32, 32, 32, 1.0, 0.0, 20.0, 0.01, 5), kw={}), precond)
    if precond == "gmg":
        assert st["levels"] >= 4 and st["iters_total"] <= 5 * 25
    # reference defaults (10^3 cells, 20 steps) with a non-zero boundary value
    okw = dict(diffusivity=1.0, T_initial=20.0, dt=0.01, num_steps=20, T_boundary=3.5)
    _check_heat(P, 3, [1, 1, 1], [10, 10, 10], okw,
                dict(args=(1, 1, 1, 10, 10, 10, 1.0, 3.5, 20.0, 0.01, 20), kw={}), precond)


@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
def test_heat_3d_directional_bcs_and_steady(P, precond):
    # directional BCs (reference :606-623) leave natural (partial-patch) faces
    for bc in (dict(T_left=10.0, T_right=1.0), dict(T_left=4.0, T_side=2.0), dict(T_side=6.0)):
        okw = dict(diffusivity=2.0, T_initial=1.0, dt=0.05, num_steps=3, **bc)
        _check_heat(P, 3, [1, 0.5, 0.25], [16, 8, 4], okw,
                    dict(args=(1, 0.5, 0.25, 16, 8, 4, 2.0, 0.0, 1.0, 0.05, 3), kw=bc), precond)
    okw = dict(diffusivity=1.5, steady=True, T_boundary=2.0, source_type="constant", source_value=50.0)
    _check_heat(P, 3, [1, 1, 1], [16, 16, 16], okw,
                dict(args=(1, 1, 1, 16, 16, 16, 1.5, 2.0, 0.0, 0.01, 5),
                     kw=dict(steady=True, source_type="constant", source_value=50.0)), precond)
    okw = dict(diffusivity=1.0, steady=True, T_left=20.0, T_right=0.0)
    f, _ = _check_heat(P, 1, [2.0], [100], okw,
                       dict(args=(2.0, 100, 1.0, 20.0, 0.0, 0.0, 0.01, 5), kw=dict(steady=True)), precond)
    x = np.asarray(f.coords)[:, 0]
    assert np.allclose(f.values[0], 20.0 * (1 - x / 2.0), atol=1e-9)   # known answer (i)


@pytest.mark.parametrize("initial_type", ["cosine", "sine"])
def test_heat_trig_initial_conditions(P, initial_type):
    # project(Expression("A*cos(k*x[0])*...", degree=2), V), reference :276-290, 408-421, 672-685
    ic = dict(initial_type=initial_type, initial_amplitude=3.0, initial_wavenumber=2.5)
    okw = dict(diffusivity=1.0, T_initial=0.0, dt=0.01, num_steps=4, T_left=1.0, T_right=0.5, **ic)
    _check_heat(P, 1, [2.0], [40], okw, dict(args=(2.0, 40, 1.0, 1.0, 0.5, 0.0, 0.01, 4), kw=ic), "jacobi")
    okw = dict(diffusivity=0.7, T_initial=0.0, dt=0.02, num_steps=3, T_boundary=0.25, **ic)
    _check_heat(P, 2, [1.0, 0.8], [20, 14], okw, dict(args=(1.0, 0.8, 20, 14, 0.7, 0.25, 0.0, 0.02, 3), kw=ic), "gmg")
    okw = dict(diffusivity=1.0, T_initial=0.0, dt=0.01, num_steps=3, T_boundary=0.0, **ic)
    _check_heat(P, 3, [1, 0.5, 0.75], [12, 6, 8], okw,
                dict(args=(1, 0.5, 0.75, 12, 6, 8, 1.0, 0.0, 0.0, 0.01, 3), kw=ic), "gmg")


# ---------------------------------------------------------------- curvilinear heat tools vs oracle LU
@pytest.mark.parametrize("kind,n,kw", [
    ("1d_cylindrical", [50], dict(r_inner=0.1, r_outer=1.0, T_inner=100.0, T_outer=20.0)),
    ("1d_cylindrical", [40], dict(r_inner=0.0, r_outer=1.0, T_inner=100.0, T_outer=20.0)),       # axis r = 0: no inner BC
    ("1d_spherical", [50], dict(r_inner=0.1, r_outer=1.0, T_inner=100.0, T_outer=20.0)),
    ("2d_cylindrical", [14, 18], dict(r_inner=0.1, r_outer=1.0, z_length=2.0, T_boundary=35.0)),
    ("2d_spherical", [12, 16], dict(r_inner=0.1, r_outer=1.0, T_boundary=35.0)),
    ("3d_spherical", [8, 7, 9], dict(r_inner=0.2, r_outer=1.0, T_boundary=35.0)),
])
@pytest.mark.parametrize("steady", [False, True])
def test_curvilinear_heat_tools(P, kind, n, kw, steady):
    common = dict(diffusivity=0.8, T_initial=20.0, dt=0.02, num_steps=4, steady=steady, source_type="constant",
                  source_value=40.0)
    ref = fo.solve_heat_curvilinear(kind, kw["r_inner"], kw["r_outer"], n, **{k: v for k, v in kw.items()
                                                                               if k not in ("r_inner", "r_outer")},
                                    **common)
    fn = getattr(P, f"_solve_heat_{kind}_raw")
    names = {"1d_cylindrical": ["nr"], "1d_spherical": ["nr"], "2d_cylindrical": ["nr", "nz"],
             "2d_spherical": ["nr", "ntheta"], "3d_spherical": ["nr", "ntheta", "nphi"]}[kind]
    f = fn(**kw, **dict(zip(names, n)), **common, as_arrays=True)
    assert f.values.shape == ref.values.shape and f.dim == ref.dim
    assert np.allclose(np.asarray(f.coords), ref.coords, rtol=0, atol=1e-14)
    assert np.allclose(f.times, ref.times, rtol=0, atol=1e-15)
    for k in range(ref.values.shape[0]):
        assert fo.rel_l2(f.values[k], ref.values[k]) <= TOL, (k, fo.rel_l2(f.values[k], ref.values[k]))
    assert P.last_stats()["converged"] == 1
    assert f.meta["coordinate_system"] in ("cylindrical", "spherical") and "r_inner" in f.meta


# ---------------------------------------------------------------- elasticity vs oracle LU
@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
@pytest.mark.parametrize("quantity", ["stress", "strain"])
def test_elasticity_3d(P, precond, quantity):
    ref = fo.solve_elasticity(3, [1, 0.2, 0.2], [40, 8, 8], 210e9, 0.3, body=[0, 0, -76518.0], quantity=quantity)
    f = P._solve_elasticity_3d_static(1, 0.2, 0.2, 40, 8, 8, 210e9, 0.3, 0.0, 0.0, -76518.0, quantity,
                                      precond=precond, as_arrays=True)
    assert np.array_equal(f.coords, ref.coords)
    err = fo.rel_l2(f.values[0], ref.values[0])
    assert err <= TOL, err
    assert P.last_stats()["converged"] == 1
    assert P.last_stats()["true_relres"] <= 1e-9, P.last_stats()


@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
def test_elasticity_displacement_and_2d_1d(P, precond):
    from pde_solver_b200 import solvers
    ref = fo.solve_elasticity(3, [1, 0.3, 0.2], [16, 6, 4], 70e9, 0.33, body=[1e4, -2e4, 3e4])
    _, val, disp = solvers._elasticity(3, [1, 0.3, 0.2], [16, 6, 4], 70e9, 0.33, [1e4, -2e4, 3e4], "stress",
                                       precond=precond, want_displacement=True)
    assert fo.rel_l2(disp, ref.aux["u"]) <= TOL
    assert fo.rel_l2(val, ref.values[0]) <= TOL
    for ps in (True, False):
        for q in ("stress", "strain"):
            ref = fo.solve_elasticity(2, [1, 0.5], [24, 12], 210e9, 0.3, body=[0, -76518.0], quantity=q,
                                      plane_stress=ps)
            f = P._solve_elasticity_2d_static(1, 0.5, 24, 12, 210e9, 0.3, 0.0, -76518.0, q, ps, precond=precond,
                                              as_arrays=True)
            assert fo.rel_l2(f.values[0], ref.values[0]) <= TOL, (ps, q)
    for q in ("stress", "strain"):
        ref = fo.solve_elasticity(1, [1.5], [64], 210e9, body=[1e6], quantity=q, area=2.0)
        f = P._solve_elasticity_1d_static(1.5, 64, 210e9, 2.0, 1e6, q, precond=precond, as_arrays=True)
        assert fo.rel_l2(f.values[0], ref.values[0]) <= TOL, q


def test_zero_body_force_gives_zero_field(P):
    f = P._solve_elasticity_3d_static(1, 1, 1, 8, 8, 8, 210e9, 0.3, as_arrays=True)    # docstring :2639-2642
    assert np.all(f.values == 0.0)


# ---------------------------------------------------------------- larger sizes: manufactured solutions
@pytest.mark.parametrize("kind,n,precond", [("heat", [128, 128, 128], "gmg"), ("heat", [96, 80, 64], "jacobi"),
                                            ("elasticity", [128, 32, 32], "gmg")])
def test_manufactured_solution_large(P, ctx, kind, n, precond):
    # (iv-c): b = A u* with the (small-size validated) GPU operator, solve, compare with u*
    L = [1.0, 1.0, 1.0] if kind == "heat" else [1.0, 0.25, 0.25]
    lam, mu = fo.lame(210e9, 0.3, 3)
    faces = {f: 0.0 for f in range(6)} if kind == "heat" else {0: 0.0}
    p = P._lib.op_params(kind, 3, n, L, 1.0, 0.01, lam, mu, bc=P._lib.make_bc(faces))
    nv, _ = P._lib.mesh_counts(3, n)
    nc = 3 if kind == "elasticity" else 1
    X = P.mesh.coordinates(3, n, L)
    mask, _ = P.mesh.dirichlet(3, n, P._lib.make_bc(faces))
    us = np.stack([np.sin(3 * X[:, 0] + c) * np.cos(2 * X[:, 1]) * (1 + X[:, 2]) for c in range(nc)])
    us[:, mask == 1] = 0.0
    b = P._lib.op_apply(ctx, p, us)
    x, st = P._lib.op_solve(ctx, p, b, P._lib.make_opts(rtol=1e-11, precond=precond))
    assert st["converged"] == 1 and st["true_relres"] < 1e-9
    assert fo.rel_l2(x, us) <= TOL, fo.rel_l2(x, us)


# ---------------------------------------------------------------- BASELINE full sizes: device-resident properties
@pytest.mark.parametrize("kind,n,L,faces", [
    ("heat", [512, 512, 512], [1.0, 1.0, 1.0], {f: 0.0 for f in range(6)}),          # config 4
    ("elasticity", [1280, 256, 256], [1.0, 0.2, 0.2], {0: 0.0}),                      # config 5
    ("heat", [4096, 4096], [1.0, 1.0], {f: 0.0 for f in range(4)}),                   # config 2
    ("elasticity", [320, 64, 64], [1.0, 0.2, 0.2], {0: 0.0}),                         # config 3
    ("heat", [333, 77, 130], [1.0, 0.3, 0.4], {0: 0.0, 3: 0.0}),                      # ragged tiles, mixed BCs
])
def test_manufactured_solution_full_size(P, ctx, kind, n, L, faces):
    # (iv-c) at the sizes BASELINE.json names: b = A u* on the device, GMG/Jacobi-PCG to rtol 1e-11, ||x-u*||/||u*||
    dim = len(n)
    lam, mu = fo.lame(210e9, 0.3, 3)
    p = P._lib.op_params(kind, dim, n, L, 1.0, 0.01, lam, mu, bc=P._lib.make_bc(faces))
    err, st = P._lib.op_manufactured(ctx, p, P._lib.make_opts(rtol=1e-11, precond="auto"))
    assert st["converged"] == 1 and st["true_relres"] < 1e-9, st
    assert err <= TOL, (err, st)


def test_multi_gpu_slabs_match_oracle():
    """2-rank slab-partitioned GMG / Jacobi heat solve against the oracle (skipped on a 1-GPU box)."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    # both halo paths: the peer-memory mailbox kernel (default) and the NCCL send/recv fallback
    for port, halo in ((29541, None), (29543, "nccl")):
        env = dict(os.environ)
        env.pop("PDE_B200_HALO", None)
        if halo:
            env["PDE_B200_HALO"] = halo
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", str(port),
                            os.path.join(root, "tests", "mgpu_check.py")], stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=600, cwd=root, env=env)
        assert r.returncode == 0 and "MGPU OK" in r.stdout, r.stdout[-3000:]
        assert "halo self-check ok" in r.stdout


# ---------------------------------------------------------------- pipelined batch of one-step advances
def test_heat_advance_batch_matches_oracle_and_serial_calls(P, ctx):
    """pde_heat_advance_batch (3-stream upload / solve / download pipeline) == set_state + step + get_state, and
    each result is one backward-Euler step of the oracle from the same input field."""
    n, L, kappa, dt = [12, 10, 9], [1.0, 0.8, 0.6], 0.7, 0.02
    m = fo.make_mesh(3, L, n)
    K, M = fo.assemble_stiffness_mass(m)
    dofs, vals = fo._merge_bcs(fo.heat_bcs(m, L, T_boundary=2.0), m.nv)
    A, _ = fo.apply_bc_rowwise((M + dt * kappa * K).tocsr(), np.zeros(m.nv), dofs, vals)
    rng = np.random.default_rng(5)
    nreq = 5
    bc = P._lib.make_bc({f: 2.0 for f in range(6)})
    for precond in ("jacobi", "gmg"):
        hs = P._lib.HeatStepper(ctx, 3, n, L, kappa, dt, T_initial=0.0, bc=bc,
                                opts=P._lib.make_opts(rtol=1e-10, precond=precond))
        assert hs.nloc == m.nv
        ins = [P._lib.PinnedArray(m.nv) for _ in range(nreq)]
        outs = [P._lib.PinnedArray(m.nv) for _ in range(nreq)]
        for a in ins:
            a.array[:] = rng.standard_normal(m.nv) * 5.0 + 3.0
        st = hs.advance_batch([a.array for a in ins], [a.array for a in outs])
        assert st["converged"] and st["solves"] == nreq
        tmp = np.empty(m.nv)
        for a, o in zip(ins, outs):
            u = a.array.copy()
            u[dofs] = vals                                   # bc.apply(u_n.vector())
            b = M @ u
            b[dofs] = vals
            ref = fo.lu_solve(A, b)
            assert np.linalg.norm(o.array - ref) <= TOL * np.linalg.norm(ref)
            hs.set_state(a.array)
            hs.step(1)
            hs.get_state(tmp)
            assert np.linalg.norm(o.array - tmp) <= 1e-12 * np.linalg.norm(tmp)
        hs.advance_batch([], [])
        hs.close()
        for a in ins + outs:
            a.free()


# ---------------------------------------------------------------- cylinder / composite-core branches of solve_heat_3D
@pytest.mark.parametrize("case", [
    dict(geometry_type="cylinder", cylinder_radius=0.3, T_boundary=1.0, T_initial=5.0, source_type="constant",
         source_value=3.0),
    dict(geometry_type="cylinder", cylinder_radius=0.3, T_left=10.0, T_right=2.0, T_side=50.0, T_initial=4.0),
    dict(geometry_type="cylinder", cylinder_radius=0.25, T_side=7.0, T_initial=4.0, source_type="constant",
         source_value=1.0),
    dict(core_radius=0.3, core_diffusivity=25.0, T_boundary=0.0, T_initial=3.0),
    dict(core_radius=0.3, core_diffusivity=25.0, T_left=1.0, T_side=2.0, T_initial=3.0),
    dict(geometry_type="cylinder", cylinder_radius=0.3, core_radius=0.15, core_diffusivity=8.0, steady=True,
         T_boundary=2.0, source_type="constant", source_value=5.0),
    dict(core_radius=0.3, core_diffusivity=4.0, T_boundary=0.5, initial_type="cosine", initial_amplitude=2.0,
         initial_wavenumber=3.0),
    dict(geometry_type="cylinder", cylinder_radius=0.3, T_boundary=0.0, initial_type="sine", initial_amplitude=1.5,
         initial_wavenumber=4.0),
    dict(geometry_type="cylinder", cylinder_radius=0.3, T_boundary=0.0, initial_type="zero", source_type="constant",
         source_value=2.0),
])
def test_heat_3d_cylinder_and_composite_core(P, case):
    Lx, Ly, Lz, n, kappa = 1.0, 0.5, 0.5, [6, 10, 10], 0.8
    kw = dict(dt=0.02, num_steps=3)
    kw.update(case)
    ref = fo.solve_heat_3d_special(Lx, Ly, Lz, n, kappa, **kw)
    args = dict(T_boundary=0.0, T_initial=0.0, steady=False)
    args.update(kw)
    f = P._solve_heat_3d_raw(Lx, Ly, Lz, n[0], n[1], n[2], kappa, args.pop("T_boundary"), args.pop("T_initial"),
                             args.pop("dt"), args.pop("num_steps"), as_arrays=True, **args)
    assert np.array_equal(np.asarray(f.coords), ref.coords)                 # shifted BoxMesh coordinates bit-exact
    v = np.asarray(f.values)
    assert v.shape == ref.values.shape
    for a, b in zip(v, ref.values):
        assert np.linalg.norm(a - b) <= TOL * max(np.linalg.norm(b), 1e-300)
    assert f.meta["geometry_type"] == case.get("geometry_type", "box")
    if "core_radius" in case:
        assert f.meta["base_diffusivity"] == kappa and "diffusivity" not in f.meta


def test_heat_solve_pinned_snapshots_pipeline(P, ctx):
    """pde_heat_solve with a PINNED values buffer: the snapshot downloads are truly asynchronous (copy stream, two
    staging slots handed over by events) and overlap the following steps; every snapshot must still be the state
    after exactly its step.  13 snapshots reuse each staging slot six times."""
    import ctypes as C
    L_ = P._lib
    n, Ld, kappa, dt, steps, stride = [20, 12, 10], [1.0, 0.6, 0.5], 0.9, 0.01, 24, 2
    ref = fo.solve_heat(3, Ld, n, kappa, T_initial=7.0, dt=dt, num_steps=steps, T_boundary=1.5,
                        source_type="constant", source_value=4.0)
    p = L_.HeatParams()
    p.dim = 3
    p.n = L_.i3(n)
    p.L = L_.d3(Ld)
    p.diffusivity, p.dt, p.num_steps, p.steady = kappa, dt, steps, 0
    p.source_value = 4.0
    p.initial_type = L_.IC["constant"]
    p.snapshot_stride = stride
    p.T_initial = 7.0
    p.bc = P.mesh.heat_bc(3, T_boundary=1.5)
    nv = ref.values.shape[1]
    nsnap = 1 + steps // stride
    buf = L_.PinnedArray(nsnap * nv)
    times = np.empty(nsnap)
    st = L_.Stats()
    o = L_.make_opts(rtol=1e-10, precond="gmg")
    try:
        buf.array[:] = np.nan
        L_.check(L_.lib().pde_heat_solve(ctx.handle, C.byref(p), C.byref(o), None, L_.ptr(buf.array), L_.ptr(times),
                                         C.byref(st)))
        vals = buf.array.reshape(nsnap, nv).copy()
    finally:
        buf.free()
    assert np.allclose(times, ref.times[::stride], rtol=0, atol=1e-15)
    for k in range(nsnap):
        assert fo.rel_l2(vals[k], ref.values[k * stride]) <= TOL, k


# ---------------------------------------------------------------- Fourier symbol of the interior stencil (SURVEY 8c iv-b)
def _symbol(dim, h, alpha, beta, theta):
    """sum_d w_d exp(i theta.d) of alpha*M + beta*K on the Kuhn / right-diagonal P1 mesh, from the closed-form weights
    (SURVEY A.2): independent of the oracle's assembly code."""
    if dim == 3:
        hx, hy, hz = h
        vol = hx * hy * hz
        kx, ky, kz = hy * hz / hx, hx * hz / hy, hx * hy / hz
        w = {(0, 0, 0): alpha * vol * 2 / 5 + beta * 2 * (kx + ky + kz)}
        for d, k in (((1, 0, 0), kx), ((0, 1, 0), ky), ((0, 0, 1), kz)):
            w[d] = alpha * vol / 20 - beta * k
        for d in ((1, 1, 0), (1, 0, 1), (0, 1, 1)):
            w[d] = alpha * vol / 30
        w[(1, 1, 1)] = alpha * vol / 20
    else:
        hx, hy = h
        vol = hx * hy
        w = {(0, 0): alpha * vol / 2 + beta * 2 * (hy / hx + hx / hy),
             (1, 0): alpha * vol / 12 - beta * hy / hx, (0, 1): alpha * vol / 12 - beta * hx / hy,
             (1, 1): alpha * vol / 12}
    zero = tuple([0] * dim)
    C = w[zero]
    for d, v in w.items():
        if d != zero:
            C += 2 * v * np.cos(np.dot(theta, d))          # the stencil is symmetric: w(-d) = w(d), the sine parts cancel
    return C, max(abs(v) for v in w.values())


@pytest.mark.parametrize("dim,n,L,faces", [(3, [512, 512, 512], [1.0, 1.0, 1.0], range(6)),          # config 4, TMA sweep
                                           (3, [320, 64, 64], [1.0, 0.2, 0.2], []),                   # config 3 grid, no BC
                                           (2, [4096, 4096], [1.0, 1.0], range(4)),                   # config 2, k_sweep2d
                                           (2, [300, 70], [1.0, 0.4], [])])                           # 2-D table kernel
def test_interior_rows_have_the_closed_form_fourier_symbol(P, ctx, dim, n, L, faces):
    """x = cos(theta.n + phi) is an eigenvector of the interior stencil with the eigenvalue sum_d w_d cos(theta.d):
    checked at the BASELINE sizes on every row whose patch is complete, against closed-form weights."""
    alpha, beta = 1.0, 0.01
    theta = np.array([0.31, 0.73, 1.17][:dim])
    nn = [k + 1 for k in n]
    ax = [np.arange(k, dtype=np.float64) for k in nn]
    phase = 0.4 + theta[0] * ax[0][None, :]                 # natural order: x fastest
    if dim == 2:
        phase = phase + theta[1] * ax[1][:, None]
    else:
        phase = phase[None, :, :] + theta[1] * ax[1][None, :, None] + theta[2] * ax[2][:, None, None]
    x = np.cos(phase)
    del phase
    h = [Lk / k for Lk, k in zip(L, n)]
    C, wmax = _symbol(dim, h, alpha, beta, theta)
    p = P._lib.op_params("heat", dim, n, L, alpha, beta, bc=P._lib.make_bc({f: 0.0 for f in faces}) if faces else None)
    y = P._lib.op_apply(ctx, p, x.reshape(1, -1)).reshape(x.shape)
    inner = tuple([slice(1, -1)] * dim)
    err = np.abs(y[inner] - C * x[inner]).max()
    assert err <= 1e-12 * 15 * wmax, (err, wmax)


# ---------------------------------------------------------------- size-independent operator properties at BASELINE sizes
@pytest.mark.parametrize("n", [[320, 64, 64], [1280, 256, 256]])
def test_elasticity_annihilates_linear_displacements_at_full_size(P, ctx, n):
    """Patch test on the GPU at the sizes of configs 3 and 5: a displacement field with a constant gradient (rigid
    motions included) has constant stress, so every row whose element patch is complete gives zero."""
    L = [1.0, 0.2, 0.2]
    lam, mu = fo.lame(210e9, 0.3, 3)
    nn = [k + 1 for k in n]
    xs = [np.linspace(0.0, Lk, k) for Lk, k in zip(L, nn)]
    G = np.array([[0.3, -1.1, 0.7], [0.9, 0.2, -0.4], [-0.6, 0.5, 1.3]])
    a0 = np.array([0.25, -0.5, 0.75])
    u = np.empty((3, nn[2], nn[1], nn[0]))
    for i in range(3):
        u[i] = a0[i] + G[i, 0] * xs[0][None, None, :] + G[i, 1] * xs[1][None, :, None] + G[i, 2] * xs[2][:, None, None]
    p = P._lib.op_params("elasticity", 3, n, L, lam=lam, mu=mu)
    scale = np.abs(P._lib.op_table(p)).max() * np.abs(u).max()
    y = P._lib.op_apply(ctx, p, u.reshape(3, -1)).reshape(u.shape)
    assert np.abs(y[:, 1:-1, 1:-1, 1:-1]).max() <= 1e-12 * scale
    assert np.abs(y).max() > 1e-6 * scale          # the traction rows on the faces are not zero


@pytest.mark.parametrize("kind,n,L,faces", [("heat", [512, 512, 512], [1.0, 1.0, 1.0], range(6)),
                                            ("elasticity", [640, 128, 128], [1.0, 0.2, 0.2], [0]),
                                            ("heat", [4096, 4096], [1.0, 1.0], range(4))])
def test_operator_is_symmetric_at_full_size(P, ctx, kind, n, L, faces):
    """x.(A y) = y.(A x) for random x, y that vanish on the Dirichlet nodes: symmetry of the matrix-free operator
    including its natural-face rows (k_face_rows) and the masked Dirichlet rows."""
    dim = len(n)
    nc = dim if kind == "elasticity" else 1
    lam, mu = fo.lame(210e9, 0.3, 3)
    bc = P._lib.make_bc({f: 0.0 for f in faces})
    mask, _ = P.mesh.dirichlet(dim, n, bc)
    free = (~mask.astype(bool)).astype(np.float64)
    rng = np.random.default_rng(3)
    x = rng.standard_normal((nc, free.size)) * free
    y = rng.standard_normal((nc, free.size)) * free
    p = P._lib.op_params(kind, dim, n, L, 1.0, 0.01, lam, mu, bc=bc)
    Ax = P._lib.op_apply(ctx, p, x)
    Ay = P._lib.op_apply(ctx, p, y)
    a, b = float(np.vdot(y, Ax)), float(np.vdot(x, Ay))
    assert abs(a - b) <= 1e-11 * max(abs(a), abs(b), float(np.linalg.norm(x) * np.linalg.norm(Ay)))
    assert float(np.vdot(x, Ax)) > 0.0               # positive definite on the free dofs


def test_null_spaces_and_volume_at_full_size(P, ctx):
    """No boundary conditions, BASELINE grids: K 1 = 0 on every row (natural-face rows included), sum(M 1) = volume,
    and the elasticity operator annihilates the six rigid-body motions on every row (traction-free faces)."""
    n, L = [512, 512, 512], [1.0, 0.7, 0.9]
    nv = 513 ** 3
    ones = np.ones((1, nv))
    pk = P._lib.op_params("stiffness", 3, n, L)
    y = P._lib.op_apply(ctx, pk, ones)
    assert np.abs(y).max() <= 1e-12 * np.abs(P._lib.op_table(pk)).max()
    pm = P._lib.op_params("mass", 3, n, L)
    y = P._lib.op_apply(ctx, pm, ones)
    assert abs(float(y.sum()) - L[0] * L[1] * L[2]) <= 1e-12
    assert y.min() > 0.0
    del y, ones
    n, L = [640, 128, 128], [1.0, 0.2, 0.2]
    lam, mu = fo.lame(210e9, 0.3, 3)
    nn = [k + 1 for k in n]
    X = [np.linspace(0.0, Lk, k) for Lk, k in zip(L, nn)]
    x = np.broadcast_to(X[0][None, None, :], nn[::-1])
    yv = np.broadcast_to(X[1][None, :, None], nn[::-1])
    z = np.broadcast_to(X[2][:, None, None], nn[::-1])
    pe = P._lib.op_params("elasticity", 3, n, L, lam=lam, mu=mu)
    cmax = np.abs(P._lib.op_table(pe)).max()
    zero = np.zeros(nn[::-1])
    one = np.ones(nn[::-1])
    modes = [(one, zero, zero), (zero, one, zero), (zero, zero, one),            # translations
             (zero, -z, yv), (z, zero, -x), (-yv, x, zero)]                      # rotations about x, y, z
    for mode in modes:
        u = np.stack([np.ascontiguousarray(c) for c in mode]).reshape(3, -1)
        r = P._lib.op_apply(ctx, pe, u)
        assert np.abs(r).max() <= 1e-12 * cmax * max(1.0, np.abs(u).max())


@pytest.mark.parametrize("precond,n,source_value", [
    ("gmg", [256, 96, 64], 0.0), ("jacobi", [64, 24, 16], 0.0),
    ("gmg", [256, 96, 64], 40.0), ("jacobi", [64, 24, 16], 40.0),
    ("gmg", [333, 77, 130], 40.0)],                    # ragged TMA tiles, face rows on the four natural faces
    ids=["gmg", "jacobi", "gmg-source", "jacobi-source", "gmg-source-ragged"])
def test_steady_heat_with_end_temperatures_is_exactly_linear(P, precond, n, source_value):
    """Known answer without the oracle: steady conduction between T_left at x = 0 and T_right at x = Lx with
    insulated (natural) side faces is linear in x, and a linear field lies in the P1 space, so the nodal values are
    exact up to the solver tolerance - on a grid far beyond what the CPU restatement can factorise.  A constant source
    f adds f x (Lx - x) / (2 kappa): the 1-D P1 solution is exact at the nodes, and the Kuhn split carries that over
    to the box (test_load_vectors.py checks the formula against the oracle), so the heat source term f m of the
    stencil kernels is checked here at full size too."""
    Lx, Ly, Lz, kappa = 2.0, 0.7, 0.5, 1.7
    f = P._solve_heat_3d_raw(Lx, Ly, Lz, n[0], n[1], n[2], kappa, 0.0, 0.0, 0.01, 1, steady=True, T_left=20.0,
                             T_right=-5.0, source_type="constant", source_value=source_value, precond=precond,
                             as_arrays=True)
    x = np.asarray(f.coords)[:, 0]
    exact = 20.0 + (-5.0 - 20.0) * x / Lx + source_value * x * (Lx - x) / (2.0 * kappa)
    u = np.asarray(f.values)[-1]
    assert np.linalg.norm(u - exact) <= TOL * np.linalg.norm(exact)
    assert P.last_stats()["converged"] == 1


def test_cylinder_branch_without_dirichlet_set_drifts_uniformly(P):
    """Known answer for the radially weighted path (n4): with T_side only, the BoxMesh 'cylinder' has no Dirichlet
    facet (reference :594-598 on a box), K_w 1 = 0 and M_w 1 = m_w, so a uniform state with a constant source f
    advances by exactly dt*f per step on every node."""
    f = P._solve_heat_3d_raw(1.0, 9.0, 9.0, 48, 60, 60, 0.9, 0.0, 4.0, 0.05, 4, source_type="constant",
                             source_value=2.5, geometry_type="cylinder", cylinder_radius=0.3, T_side=7.0,
                             as_arrays=True)
    v = np.asarray(f.values)
    assert v.shape == (5, 49 * 37 * 37)
    for k in range(5):
        assert np.abs(v[k] - (4.0 + k * 0.05 * 2.5)).max() <= 1e-8 * 4.0


@pytest.mark.parametrize("nx,precond", [(100, "jacobi"), (4096, "gmg"), (100000, "gmg")])
def test_heat_1d_sine_mode_decays_by_the_closed_form_factor(P, nx, precond):
    """(iv-a) on the GPU: sin(j pi x / L) at the nodes is an eigenvector of M = h/6 [1 4 1] and K = 1/h [-1 2 -1]
    under homogeneous Dirichlet conditions, so every backward-Euler step multiplies it by lam_M / (lam_M + dt k lam_K)."""
    L, dt, kappa, j, steps = 2.0, 0.01, 1.3, 3, 5
    h = L / nx
    x = np.arange(nx + 1) * h
    u0 = np.sin(j * np.pi * x / L)
    u0[0] = u0[-1] = 0.0
    th = j * np.pi * h / L
    lamM, lamK = h / 6 * (4 + 2 * np.cos(th)), (2 - 2 * np.cos(th)) / h
    g = lamM / (lamM + dt * kappa * lamK)
    f = P._solve_heat_1d_raw(L, nx, kappa, 0.0, 0.0, 0.0, dt, steps, u0=u0, precond=precond, as_arrays=True)
    v = np.asarray(f.values)
    for k in range(steps + 1):
        assert np.linalg.norm(v[k] - g ** k * u0) <= TOL * np.linalg.norm(u0), k


def test_elasticity_scaling_laws(P):
    """Linearity at a size the oracle cannot reach: the projected von Mises stress is proportional to the body
    force and independent of E; the von Mises strain is proportional to the force and to 1/E."""
    args = (1.0, 0.2, 0.2, 160, 32, 32)
    s1 = np.asarray(P._solve_elasticity_3d_static(*args, 210e9, 0.3, 0.0, 0.0, -76518.0, "stress", as_arrays=True).values[0])
    s2 = np.asarray(P._solve_elasticity_3d_static(*args, 210e9, 0.3, 0.0, 0.0, -3 * 76518.0, "stress", as_arrays=True).values[0])
    s3 = np.asarray(P._solve_elasticity_3d_static(*args, 70e9, 0.3, 0.0, 0.0, -76518.0, "stress", as_arrays=True).values[0])
    e1 = np.asarray(P._solve_elasticity_3d_static(*args, 210e9, 0.3, 0.0, 0.0, -76518.0, "strain", as_arrays=True).values[0])
    e3 = np.asarray(P._solve_elasticity_3d_static(*args, 70e9, 0.3, 0.0, 0.0, -76518.0, "strain", as_arrays=True).values[0])
    assert s1.max() > 1e5
    assert fo.rel_l2(s2, 3.0 * s1) <= 10 * TOL
    assert fo.rel_l2(s3, s1) <= 10 * TOL
    assert fo.rel_l2(e3, 3.0 * e1) <= 10 * TOL


def test_heat_superposition_at_128_cubed(P):
    """The backward-Euler map is affine in (initial value, boundary value, source): the solve with all three equals
    the sum of the solves with the initial value alone and with boundary value + source alone (2.1 M dofs, GMG-PCG)."""
    g = (1.0, 1.0, 1.0, 128, 128, 128, 0.8)
    a = np.asarray(P._solve_heat_3d_raw(*g, 0.0, 20.0, 0.01, 3, precond="gmg", as_arrays=True).values)
    b = np.asarray(P._solve_heat_3d_raw(*g, 5.0, 0.0, 0.01, 3, source_type="constant", source_value=3.0, precond="gmg",
                                        as_arrays=True).values)
    c = np.asarray(P._solve_heat_3d_raw(*g, 5.0, 20.0, 0.01, 3, source_type="constant", source_value=3.0,
                                        precond="gmg", as_arrays=True).values)
    # the boundary nodes of the initial snapshot carry T_boundary in every run: a has 0 there, b has 5, c has 5
    for k in range(1, 4):
        assert fo.rel_l2(c[k], a[k] + b[k]) <= 10 * TOL, k


def test_dof_permutation_reorders_exports(P):
    """Row a3: with a dof numbering plugged in (as DOLFIN's reorder_dofs_serial=True would give), coordinates, values,
    cell-dof tables and Dirichlet masks leave in that numbering, still paired node by node."""
    n, L = [6, 5], [1.0, 0.6]
    rng = np.random.default_rng(3)
    nv = 7 * 6
    perm = rng.permutation(nv)
    base = P._solve_heat_2d_raw(1.0, 0.6, 6, 5, 1.0, 0.0, 20.0, 0.01, 3, as_arrays=True)
    cd0 = P.mesh.cell_dofs(2, n)
    m0, _ = P.mesh.dirichlet(2, n, P._lib.make_bc({f: 0.0 for f in range(4)}))
    P.mesh.set_dof_permutation(2, n, perm)
    try:
        f = P._solve_heat_2d_raw(1.0, 0.6, 6, 5, 1.0, 0.0, 20.0, 0.01, 3, as_arrays=True)
        assert np.array_equal(f.coords, base.coords[perm]) and np.array_equal(f.values, base.values[:, perm])
        cd = P.mesh.cell_dofs(2, n)
        assert np.array_equal(perm[cd], cd0)                  # dof -> vertex through the plugged map gives the natural table
        m1, _ = P.mesh.dirichlet(2, n, P._lib.make_bc({f: 0.0 for f in range(4)}))
        assert np.array_equal(m1, m0[perm])
    finally:
        P.mesh.set_dof_permutation(2, n, None)


# ---------------------------------------------------------------- the MCP tools on several GPUs from ONE process
def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_mcp_tools_use_two_gpus_from_one_process(monkeypatch, tmp_path):
    """PDE_B200_GPUS=2: solve_heat_3D / solve_elasticity_3D_static (the functions the orchestrator calls in its single
    tool process, multi_agent_orchestrator.py:70-78) run slab-partitioned on two GPUs through spawned worker ranks and
    return the single-GPU arrays."""
    import pickle

    import fenics_mcp_server as srv
    monkeypatch.setenv("PDE_B200_GPUS", "2")
    r = srv.solve_heat_3D(1.0, 1.0, 0.5, 32, 32, 16, 1.0, 0.0, 20.0, 0.01, 3, data_dir=str(tmp_path))
    f = pickle.load(open(r.data_file, "rb"))
    ref = fo.solve_heat(3, [1, 1, 0.5], [32, 32, 16], 1.0, T_initial=20.0, dt=0.01, num_steps=3)
    assert np.array_equal(np.asarray(f.coords), ref.coords)
    for k in range(4):
        assert fo.rel_l2(np.asarray(f.values[k]), ref.values[k]) <= TOL
    import pde_solver_b200 as P
    assert P.last_stats().get("gpus") == 2
    r = srv.solve_elasticity_3D_static(1.0, 0.2, 0.2, 40, 8, 8, 210e9, 0.3, 0.0, 0.0, -76518.0, "stress",
                                       data_dir=str(tmp_path))
    g = pickle.load(open(r.data_file, "rb"))
    ref2 = fo.solve_elasticity(3, [1, 0.2, 0.2], [40, 8, 8], 210e9, 0.3, body=[0, 0, -76518.0])
    assert fo.rel_l2(np.asarray(g.values[0]), ref2.values[0]) <= TOL
    assert P.last_stats().get("gpus") == 2
    from pde_solver_b200 import multi
    multi.pool().close()
