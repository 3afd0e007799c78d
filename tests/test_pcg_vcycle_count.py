"""GMG-PCG tests convergence before the V-cycle, as oracle.gmg_model.pcg does, so a solve of k iterations runs k V-cycles.

pde_stats.precond_applies counts the V-cycles of a call: one before the loop and one in every iteration that goes on,
none when the start already meets rtol.  The iteration that converges only adds alpha p to x.  That last step is about
rtol of x, far below the solution bars of the other tests, so the solution after k iterations is compared with the
model's after exactly k iterations."""
import ctypes as C

import numpy as np
import pytest

import test_vcycle_parity as vp
from oracle import gmg_model as gm

CASES = ["heat3d_128", "heat3d_128_xends", "elast3d_64"]
# max|x - x_model| / max|x_model| after the GPU's k iterations (11 on both heat cases): 3.5e-14 measured on a B200
# (power limit 1000 W).  The last x += alpha p is 5.9e-10 / 2.6e-10 of x there, and a library built without it fails
# this bar by that much.  elast3d_64 is left out: after its 29 iterations x is 1.2e-11 away from the model's, a third
# of its last step (4.1e-11).
X_CASES = ["heat3d_128", "heat3d_128_xends"]
BAR = 1e-12


@pytest.fixture(scope="module")
def P():
    import pde_solver_b200 as p
    return p


@pytest.fixture(scope="module")
def ctx(P):
    return P._lib.default_context()


def op_solve(P, ctx, name, b, **opts):
    """(x [ncomp * nverts], raw pde_stats) of a GMG op_solve of a test_vcycle_parity case"""
    L = P._lib
    b = np.ascontiguousarray(b.reshape(vp.ncomp(name), -1), dtype=np.float64)
    x = np.empty_like(b)
    st = L.Stats()
    o = L.make_opts(precond="gmg", check_every=1, **opts)
    L.check(L.lib().pde_op_solve(ctx.handle, C.byref(vp.op_params(P, name)), C.byref(o), L.ptr(b), L.ptr(x),
                                 C.byref(st)))
    return x.ravel(), st


def model_levels(P, ctx, name):
    levels, _ = vp.model(name)
    if vp.ncomp(name) > 1:      # the model smooths with the GPU's power-iteration bounds (as test_vcycle_parity)
        levels = vp.with_lmax(levels, vp.gpu_vcycle(P, ctx, name)[4]["lmax"])
    return levels


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_op_solve_runs_one_vcycle_per_iteration(P, ctx, name):
    _, st = op_solve(P, ctx, name, vp.rhs(name, seed=3), rtol=1e-10)
    assert st.converged == 1 and st.iters_total > 0
    assert st.precond_applies == st.iters_total, (st.precond_applies, st.iters_total)


@pytest.mark.gpu
@pytest.mark.parametrize("name", X_CASES)
def test_op_solve_x_is_the_models_after_k_iterations(P, ctx, name):
    b = vp.rhs(name, seed=3)
    x, st = op_solve(P, ctx, name, b, rtol=1e-10)
    k = int(st.iters_total)
    levels = model_levels(P, ctx, name)
    xm, _ = gm.pcg(levels, b, rtol=0.0, max_iters=k)
    xm1, _ = gm.pcg(levels, b, rtol=0.0, max_iters=k - 1)
    scale = np.abs(xm).max()
    ratio = np.abs(x - xm).max() / scale
    last = np.abs(xm - xm1).max() / scale
    print(f"[pcg x] {name}: k = {k}, max|x - x_model| / max|x_model| = {ratio:.2e}, last step {last:.2e}")
    assert last >= 10 * BAR, last       # the bar sees a missing last x += alpha p
    assert ratio <= BAR, ratio


def heat_stepper(P, ctx, steady, rtol, T_initial=20.0):
    n = [64, 64, 64]
    bc = P._lib.make_bc({f: 35.0 for f in range(6)})
    return P._lib.HeatStepper(ctx, 3, n, [1.0, 1.0, 1.0], 0.8, 0.01, T_initial=T_initial, bc=bc, source_value=40.0,
                              steady=steady, opts=P._lib.make_opts(rtol=rtol, precond="gmg"))


def heat_step(P, hs, nsteps):
    st = P._lib.Stats()
    P._lib.check(P._lib.lib().pde_heat_step(hs.handle, nsteps, C.byref(st)))
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("steady", [False, True], ids=["transient", "steady"])
def test_heat_stepper_runs_one_vcycle_per_iteration(P, ctx, steady):
    """The heat step takes r0.r0 for the first convergence test from its right-hand-side pass."""
    nsteps = 1 if steady else 3
    hs = heat_stepper(P, ctx, steady, 1e-10)
    try:
        st = heat_step(P, hs, nsteps)
    finally:
        hs.close()
    assert st.converged == 1 and st.levels >= 3 and st.solves == nsteps
    assert st.iters_total >= 3 * nsteps, st.iters_total
    assert st.precond_applies == st.iters_total, (st.precond_applies, st.iters_total)


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["op_solve", "heat_transient", "heat_steady"])
def test_start_that_meets_rtol_runs_no_vcycle(P, ctx, what):
    if what == "op_solve":
        # r0 = b here; r0.r0 and ||b||^2 are summed by different kernels, so rtol sits just above 1
        x, st = op_solve(P, ctx, "heat3d_128", vp.rhs("heat3d_128", seed=3), rtol=1.0 + 1e-9)
        assert not x.any()
    else:
        # steady: ||b||^2 is r0.r0.  Transient from u_n = 35 everywhere (the boundary value): K u_n = 0, so
        # r0 = dt f m, about 1 % of b = M u_n + dt f m = (35 + dt f) m
        hs = heat_stepper(P, ctx, what == "heat_steady", 1.0, T_initial=35.0)
        try:
            st = heat_step(P, hs, 1)
        finally:
            hs.close()
    assert st.converged == 1 and st.solves == 1 and st.levels >= 3
    assert st.iters_total == 0 and st.precond_applies == 0, (st.iters_total, st.precond_applies)


@pytest.mark.gpu
def test_weighted_solve_runs_one_vcycle_per_iteration(P, ctx):
    """Three backward-Euler steps of the 2-D spherical weighted operator with its Galerkin hierarchy (wmg_pcg)."""
    L = P._lib
    p = L.WheatParams()
    p.dim, p.n, p.lo, p.hi = 2, L.i3([64, 64]), L.d3([0.1, 0.0], 0.0), L.d3([1.0, np.pi], 1.0)
    p.weight_rpow, p.weight_sin_axis1, p.weight_degree = 2, 1, 2
    p.diffusivity, p.dt, p.num_steps, p.snapshot_stride = 0.8, 0.01, 3, 1
    p.source_value, p.T_initial = 40.0, 20.0
    p.bc = L.make_bc({f: 35.0 for f in range(4)})
    nv, _ = L.mesh_counts(2, [64, 64])
    values, times = np.empty((4, nv)), np.empty(4)
    st = L.Stats()
    o = L.make_opts(rtol=1e-10, precond="gmg")
    L.check(L.lib().pde_wheat_solve(ctx.handle, C.byref(p), C.byref(o), L.ptr(values), L.ptr(times), C.byref(st)))
    assert st.converged == 1 and st.levels >= 3 and st.solves == 3
    assert st.iters_total >= 3, st.iters_total
    assert st.precond_applies == st.iters_total, (st.precond_applies, st.iters_total)
