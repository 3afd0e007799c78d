"""The multigrid V-cycle on the GPU against the NumPy V-cycle of oracle.gmg_model, cycle by cycle.

A wrong preconditioner does not make PCG wrong, only slower, so the solution tests cannot see it.  The V-cycle is a
fixed linear map z = B b; pde_op_vcycle applies the solver's own hierarchy to a host vector and returns B b.

CPU part: the model itself (B symmetric and positive, P^T equal to the restriction formula of k_restrict and the
residual-restriction mode of k_heat_post2).  GPU part: B b against the model at every size the model can build, with
info.paths pinning which fused kernels each case runs; the kernel variants behind the environment switches (each in a
subprocess: the switches are read once per process); the PCG iteration count against the model; symmetry,
positivity and graph-replay repeatability at the benchmark sizes."""
import copy
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import fem_oracle as fo
from oracle import gmg_model as gm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALPHA, BETA = 1.0, 0.013
LAME = fo.lame(210e9, 0.3, 3)
# max|z - z_model| <= BAR * max|z_model|; worst measured on a B200: 1.7e-13 (elasticity 64x16x16), heat <= 3.6e-15
BAR = 2e-11
FIRST2, HEAT_POST2, POST2_R1, RR = 1, 2, 4, 8


def dirichlet_pred(L, faces, side_excl=False):
    """Dirichlet vertices of make_bc(faces): face f = 2 axis + (0: low, 1: high); side_excl: the faces of the other
    axes skip the x-ends (the reference's other_faces predicate)."""
    def pred(X, n):
        sel = np.zeros(X.shape[0], bool)
        xend = fo.near(X[:, 0], 0.0) | fo.near(X[:, 0], L[0])
        for f in faces:
            ax, hi = divmod(f, 2)
            on = fo.near(X[:, ax], L[ax] if hi else 0.0)
            if side_excl and ax > 0:
                on &= ~xend
            sel |= on
        return sel
    return pred


ALL = lambda dim: tuple(range(2 * dim))   # noqa: E731
CASES = {
    # level 0: 129 x 65 x 65 nodes, CW = 64 tiles (last x tile 5 columns, last y tile one row); levels 1-2: CW = 32
    # post2 + RR; then the generic kernels, dense coarsest level, graph
    "heat3d_128": dict(kind="heat", dim=3, n=(128, 64, 64), faces=ALL(3)),
    # 121 / 61 nodes: CW = 32 with a one-column last x tile; coarsest 31 x 11 x 10 nodes, smoothed; graph
    "heat3d_120": dict(kind="heat", dim=3, n=(120, 40, 36), faces=ALL(3)),
    # two levels, smoothed coarsest, no graph
    "heat3d_130": dict(kind="heat", dim=3, n=(130, 40, 36), faces=ALL(3)),
    # non-uniform diagonals: k_cheby_first, face rows, separate residual + k_restrict
    "heat3d_128_xends": dict(kind="heat", dim=3, n=(128, 64, 64), faces=(0, 1)),
    "heat3d_128_natural": dict(kind="heat", dim=3, n=(128, 64, 64), faces=()),
    "heat3d_128_sides": dict(kind="heat", dim=3, n=(128, 64, 64), faces=(2, 3, 4, 5), side_excl=True),
    # one level: the nl == 1 smoothing with the dot slot
    "heat3d_63": dict(kind="heat", dim=3, n=(63, 40, 36), faces=ALL(3)),
    "heat2d_256": dict(kind="heat", dim=2, n=(256, 128), faces=ALL(2)),
    "heat2d_256_xends": dict(kind="heat", dim=2, n=(256, 128), faces=(0, 1)),
    "heat1d_4096": dict(kind="heat", dim=1, n=(4096,), faces=(0, 1)),
    "heat1d_100": dict(kind="heat", dim=1, n=(100,), faces=(0, 1)),
    # k_elast3d FIRST2, face tiles, NC = 3 transfers, dense and smoothed coarsest levels
    "elast3d_64": dict(kind="elasticity", dim=3, n=(64, 16, 16), faces=(0,)),
    "elast3d_66": dict(kind="elasticity", dim=3, n=(66, 20, 12), faces=(0, 3, 4)),
    "elast2d_64": dict(kind="elasticity", dim=2, n=(64, 16), faces=(0,)),
}


def length(dim):
    return [1.0, 0.6, 0.35][:dim]


@functools.lru_cache(maxsize=None)
def model(name):
    """(levels, free mask [ncomp * nverts]) of the model hierarchy of a case (built once per module)."""
    c = CASES[name]
    dim, L = c["dim"], length(c["dim"])
    el = LAME if c["kind"] == "elasticity" else None
    levels = gm.build(dim, L, list(c["n"]), ALPHA, BETA, dirichlet_pred(L, c["faces"], c.get("side_excl", False)),
                      elasticity=el)
    return levels, levels[0].free


def rhs(name, seed=0):
    levels, free = model(name)
    return np.random.default_rng(seed).standard_normal(free.size) * free


def with_lmax(levels, lmax):
    out = []
    for lv, v in zip(levels, lmax):
        lv = copy.copy(lv)
        lv.lmax = v
        out.append(lv)
    return out


def model_z(name, b, lmax=None, nu=2):
    """B b of the model; lmax: per-level Chebyshev bounds to use instead of the model's own."""
    levels, _ = model(name)
    if lmax is not None:
        levels = with_lmax(levels, lmax)
    return gm.vcycle(levels, b, nu=nu)


def expected_paths(name, nl, n_dense, nu=2):
    """PDE_MG_* bits each level of a case must report (default kernels)."""
    c = CASES[name]
    uniform = c["kind"] == "heat" and set(c["faces"]) == set(ALL(c["dim"])) and not c.get("side_excl")
    out = []
    for l in range(nl):
        smoothed = not (l == nl - 1 and n_dense > 0)
        sweeps = nu if (l < nl - 1 or nl == 1) else 8          # the coarsest of several levels: 8 sweeps
        bits = 0
        if smoothed and uniform and sweeps >= 2:
            bits |= FIRST2
        if c["kind"] == "elasticity" and c["dim"] == 3 and l == 0 and sweeps >= 2:
            bits |= FIRST2
        if uniform and c["dim"] == 3 and l < nl - 1:
            nodes = [k // 2 ** l + 1 for k in c["n"]]
            if nodes[0] >= 32 and nodes[1] >= 8 and nodes[2] >= 8:
                bits |= RR | (HEAT_POST2 if nu == 2 else 0)
        out.append(bits)
    return out


# ---------------------------------------------------------------- CPU: the model
@pytest.mark.parametrize("name", ["heat3d_120", "heat3d_63", "elast3d_64"])
def test_model_vcycle_is_symmetric_and_positive(name):
    _, free = model(name)
    rng = np.random.default_rng(5)
    u, v = (rng.standard_normal(free.size) * free for _ in range(2))
    Bu, Bv = model_z(name, u), model_z(name, v)
    assert abs(u @ Bv - v @ Bu) <= 1e-13 * np.linalg.norm(u) * np.linalg.norm(Bv)
    assert u @ Bu > 0 and v @ Bv > 0


@pytest.mark.parametrize("n", [(6, 4, 4), (6, 4), (8,)])
def test_model_restriction_is_the_kuhn_neighbour_formula(n):
    """P^T r at coarse node X = r(2X) + 1/2 sum of r over the 14 / 6 / 2 Kuhn neighbours 2X +- p (p in {0,1}^dim \\ 0),
    the formula of k_restrict and of the residual-restriction mode of k_heat_post2."""
    dim = len(n)
    nnf = [k + 1 for k in n]
    nnc = [k // 2 + 1 for k in n]
    R = np.zeros((int(np.prod(nnc)), int(np.prod(nnf))))
    flat = lambda I, nn: sum(I[q] * int(np.prod(nn[:q])) for q in range(dim))   # noqa: E731
    ps = [p for p in np.ndindex(*([2] * dim)) if any(p)]
    assert len(ps) == 2 ** dim - 1
    for X in np.ndindex(*nnc[::-1]):
        X = X[::-1]
        i = flat(X, nnc)
        R[i, flat([2 * x for x in X], nnf)] += 1.0
        for p in ps:
            for s in (1, -1):
                F = [2 * X[q] + s * p[q] for q in range(dim)]
                if all(0 <= F[q] < nnf[q] for q in range(dim)):
                    R[i, flat(F, nnf)] += 0.5
    P = gm.prolongation(list(n) + [0] * (3 - dim))
    assert np.array_equal(P.T.toarray(), R)


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def P():
    import pde_solver_b200 as p
    return p


@pytest.fixture(scope="module")
def ctx(P):
    return P._lib.default_context()


def op_params(P, name):
    c = CASES[name]
    dim = c["dim"]
    lam, mu = LAME
    return P._lib.op_params(c["kind"], dim, list(c["n"]), length(dim), ALPHA, BETA, lam, mu,
                            bc=P._lib.make_bc({f: 0.0 for f in c["faces"]}, c.get("side_excl", False)))


def ncomp(name):
    return CASES[name]["dim"] if CASES[name]["kind"] == "elasticity" else 1


_GPU = {}


def gpu_vcycle(P, ctx, name, nu=2):
    key = (name, nu)
    if key not in _GPU:
        b = rhs(name)
        opts = P._lib.make_opts(precond="gmg", cheby_degree=nu)
        z1, z3, bz, info = P._lib.op_vcycle(ctx, op_params(P, name), b.reshape(ncomp(name), -1), opts, ncycles=3)
        _GPU[key] = (b, z1.ravel(), z3.ravel(), bz, info)
    return _GPU[key]


def check_against_model(name, b, z1, z3, bz, info, nu=2, graph=True):
    """The checks every V-cycle case makes; returns max|z - z_model| / max|z_model|."""
    levels, free = model(name)
    nl = len(levels)
    assert info["levels"] == nl
    assert info["n"] == [lv.n + [0] * (3 - len(lv.n)) for lv in levels]
    assert info["n_dense"] == (levels[-1].idx.size if levels[-1].dense is not None else 0)
    if ncomp(name) > 1:
        # the power estimate of lmax(D^-1 A) from the GPU's start vector, then the model cycles with the GPU's bounds
        for l, lv in enumerate(levels):
            assert abs(info["lmax"][l] - lv.lmax) <= 1e-10 * lv.lmax, (l, info["lmax"][l], lv.lmax)
        ref = model_z(name, b, info["lmax"], nu)
    else:
        for l, lv in enumerate(levels):
            if not (l == nl - 1 and lv.dense is not None):   # the dense coarsest level smooths nothing
                assert abs(info["lmax"][l] - lv.lmax) <= 1e-14 * lv.lmax, (l, info["lmax"][l], lv.lmax)
        ref = model_z(name, b, None, nu)
    ratio = np.abs(z1 - ref).max() / np.abs(ref).max()
    print(f"[vcycle] {name} nu={nu} levels={nl} max|z-z_model|/max|z_model| = {ratio:.2e}")
    assert ratio <= BAR, ratio
    assert not z1[~free].any()
    assert np.array_equal(z3, z1)
    assert info["graph"] == (1 if graph and nl >= 3 else 0)
    assert abs(bz - b @ z1) <= 1e-12 * np.abs(b * z1).sum()
    return ratio


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_vcycle_matches_model(P, ctx, name):
    b, z1, z3, bz, info = gpu_vcycle(P, ctx, name)
    check_against_model(name, b, z1, z3, bz, info)
    assert info["paths"] == expected_paths(name, info["levels"], info["n_dense"]), info["paths"]


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [1, 3])
def test_vcycle_other_smoother_degrees_match_model(P, ctx, nu):
    """nu = 1: no fused first sweeps, no post2; nu = 3: the sweep that rebuilds d from x1 = s0 D^-1 b (prev_mode 3)."""
    name = "heat3d_128"
    b, z1, z3, bz, info = gpu_vcycle(P, ctx, name, nu)
    check_against_model(name, b, z1, z3, bz, info, nu=nu)
    assert info["paths"] == expected_paths(name, info["levels"], info["n_dense"], nu), info["paths"]


_SUB = r"""
import json, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import pde_solver_b200 as P
from test_vcycle_parity import op_params, ncomp
ctx = P._lib.default_context()
out = sys.argv[2]
for name in sys.argv[3:]:
    b = np.load(f"{out}/{name}_b.npy")
    z1, z3, bz, info = P._lib.op_vcycle(ctx, op_params(P, name), b.reshape(ncomp(name), -1),
                                        P._lib.make_opts(precond="gmg"), ncycles=3)
    np.save(f"{out}/{name}_z1.npy", z1.ravel())
    np.save(f"{out}/{name}_z3.npy", z3.ravel())
    with open(f"{out}/{name}_info.json", "w") as f:
        json.dump(dict(info, bz=bz), f)
"""

VARIANTS = {
    "no_rr": {"PDE_B200_NO_RR": "1"},
    "no_heat2": {"PDE_B200_NO_HEAT2": "1"},                    # k_post2 + separate residual and restriction
    "no_post2": {"PDE_B200_NO_HEAT2": "1", "PDE_B200_NO_POST2": "1"},
    "cw32": {"PDE_B200_P2_CW": "32"},
    "cw64_ysb3": {"PDE_B200_P2_CW": "64", "PDE_B200_P2_YSB": "3"},
    "zc5": {"PDE_B200_P2_ZC": "5"},                            # odd z-chunk starts
    "no_graph": {"PDE_B200_MG_GRAPH": "0"},
    "no_sweep": {"PDE_B200_NO_SWEEP": "1"},
}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_kernel_variants_match_model_and_default(P, ctx, variant, tmp_path):
    names = ["heat3d_128", "heat3d_120"]
    for name in names:
        np.save(tmp_path / f"{name}_b.npy", rhs(name))
    env = dict(os.environ, **VARIANTS[variant])
    r = subprocess.run([sys.executable, "-c", _SUB, ROOT, str(tmp_path)] + names, env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    for name in names:
        b = rhs(name)
        z1, z3 = np.load(tmp_path / f"{name}_z1.npy"), np.load(tmp_path / f"{name}_z3.npy")
        with open(tmp_path / f"{name}_info.json") as f:
            info = json.load(f)
        check_against_model(name, b, z1, z3, info["bz"], info, graph=variant != "no_graph")
        _, z_def, _, _, info_def = gpu_vcycle(P, ctx, name)
        assert np.abs(z1 - z_def).max() <= 1e-12 * np.abs(z_def).max()
        p, p_def = info["paths"], info_def["paths"]
        post = HEAT_POST2 | POST2_R1
        if variant == "no_rr":
            assert p[0] == p_def[0] & ~RR and p_def[0] & RR
        elif variant == "no_heat2":
            assert p[0] == (p_def[0] & ~(RR | post)) | POST2_R1 and p_def[0] & HEAT_POST2
        elif variant == "no_post2":
            assert p[0] == p_def[0] & ~(RR | post)
        else:
            assert p == p_def


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["heat3d_128", "heat3d_128_xends", "elast3d_64"])
def test_pcg_iterations_match_model(P, ctx, name):
    """GMG-PCG takes the model's number of iterations (within one) at rtol 1e-10."""
    b = rhs(name, seed=3)
    opts = P._lib.make_opts(rtol=1e-10, precond="gmg", check_every=1)
    _, st = P._lib.op_solve(ctx, op_params(P, name), b.reshape(ncomp(name), -1), opts)
    assert st["converged"] == 1
    levels, _ = model(name)
    if ncomp(name) > 1:
        levels = with_lmax(levels, gpu_vcycle(P, ctx, name)[4]["lmax"])
    _, hist = gm.pcg(levels, b, rtol=1e-10, max_iters=200)
    assert hist[-1] <= 1e-10
    print(f"[pcg] {name}: GPU {st['iters_total']} iterations, model {len(hist)}")
    assert abs(st["iters_total"] - len(hist)) <= 1, (st["iters_total"], len(hist))


FULL = [("heat", 3, [512, 512, 512], [1.0, 1.0, 1.0], None),
        ("heat", 2, [4096, 4096], [1.0, 1.0], None),
        ("elasticity", 3, [640, 128, 128], [1.0, 0.2, 0.2], {0: 0.0})]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dim,n,L,faces", FULL)
def test_vcycle_symmetric_positive_repeatable_at_full_size(P, ctx, kind, dim, n, L, faces):
    """The bench.py workloads, where the model cannot run: u.Bv = v.Bu, u.Bu > 0, the replayed graph cycle repeats the
    live one bit for bit; on 512^3 level 0 runs the fused kernels the benchmark times."""
    faces = faces if faces is not None else {f: 0.0 for f in range(2 * dim)}
    lam, mu = LAME
    p = P._lib.op_params(kind, dim, n, L, ALPHA, BETA, lam, mu, bc=P._lib.make_bc(faces))
    nc = dim if kind == "elasticity" else 1
    mask, _ = P.mesh.dirichlet(dim, n, P._lib.make_bc(faces))
    free = mask == 0
    opts = P._lib.make_opts(precond="gmg")
    rng = np.random.default_rng(7)
    u = rng.standard_normal((nc, free.size)) * free
    Bu, Bu3, _, info = P._lib.op_vcycle(ctx, p, u, opts, ncycles=3)
    assert np.array_equal(Bu3, Bu)
    del Bu3
    v = rng.standard_normal((nc, free.size)) * free
    Bv, Bv3, _, _ = P._lib.op_vcycle(ctx, p, v, opts, ncycles=3)
    assert np.array_equal(Bv3, Bv)
    del Bv3
    uBv, vBu = np.vdot(u, Bv), np.vdot(v, Bu)
    defect = abs(uBv - vBu) / (np.linalg.norm(u) * np.linalg.norm(Bv))
    print(f"[vcycle] {kind} {n}: levels {info['levels']}, |u.Bv - v.Bu| / (|u||Bv|) = {defect:.2e}")
    assert defect <= 1e-11
    assert np.vdot(u, Bu) > 0 and np.vdot(v, Bv) > 0
    assert info["graph"] == 1
    if dim == 3 and kind == "heat":
        assert info["paths"][0] == FIRST2 | HEAT_POST2 | RR
