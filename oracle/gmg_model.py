"""NumPy model of the GPU solver's geometric-multigrid PCG (test infrastructure / tuning aid).

Mirrors pde_solver_b200/csrc/solver.cu: Kuhn edge-midpoint prolongation, R = P^T, rediscretised
coarse operators, Chebyshev(Jacobi) smoother with the Gershgorin bound (vector operators: the power
estimate of estimate_lmax), dense coarsest solve.  Vector (elasticity) levels use the blocked dof
layout [c][v] of the C ABI, P (x) I and point-Jacobi with the assembled diagonal."""
import numpy as np
import scipy.sparse as sp

from . import fem_oracle as fo


def prolongation(nf, dim=3):
    nf = list(nf) + [0] * (3 - len(nf))
    nc = [k // 2 for k in nf]
    nnf = [k + 1 for k in nf]
    nnc = [k + 1 for k in nc]
    K, J, I = np.meshgrid(np.arange(nnf[2]), np.arange(nnf[1]), np.arange(nnf[0]), indexing="ij")
    I, J, K = I.ravel(), J.ravel(), K.ravel()
    px, py, pz = I & 1, J & 1, K & 1
    lo = (I - px) // 2 + nnc[0] * ((J - py) // 2 + nnc[1] * ((K - pz) // 2))
    hi = (I + px) // 2 + nnc[0] * ((J + py) // 2 + nnc[1] * ((K + pz) // 2))
    f = np.arange(I.size)
    return sp.csr_matrix((np.full(2 * f.size, 0.5), (np.concatenate([f, f]), np.concatenate([lo, hi]))),
                         shape=(f.size, int(np.prod(nnc))))


class Level:
    pass


def power_lmax(lv, iters=12):
    """estimate_lmax of solver.cu: min(Gershgorin bound, 1.1 * the power estimate of lmax(D^-1 A)) after `iters` steps
    from the GPU's start vector sin(0.37 (node mod 1000003) + comp) + 0.5 on the free dofs (k_fill_pattern)."""
    nv = lv.A.shape[0] // lv.ncomp
    node = np.tile(np.arange(nv), lv.ncomp)
    comp = np.repeat(np.arange(lv.ncomp), nv)
    x = np.where(lv.free, np.sin(0.37 * (node % 1000003) + comp) + 0.5, 0.0)
    lam = 0.0
    for _ in range(iters):
        y = lv.dinv * (lv.Am @ x)
        yy, xx = y @ y, x @ x
        if not (yy > 0 and xx > 0):
            break
        lam = np.sqrt(yy / xx)
        x = y / np.sqrt(yy)
    return min(lv.lmax, 1.1 * lam) if lam > 0 else lv.lmax


def build(dim, L, n, alpha, beta, dir_pred, max_levels=99, dense_max=768, elasticity=None, lmax=None):
    """Scalar operator alpha*M + beta*K, or with elasticity=(lam, mu) the elasticity operator (dim components, blocked
    dofs, every component fixed on a Dirichlet vertex, at least 2 cells per axis on every coarse level);
    dir_pred(coords, n)->bool mask of Dirichlet vertices.  lmax: the Chebyshev upper bound of each level (e.g. what
    the GPU reports) instead of the model's own."""
    levels = []
    n = list(n)
    ncomp = dim if elasticity is not None else 1
    min_cells = 2 if ncomp > 1 else 1
    while True:
        m = fo.make_mesh(dim, L, n)
        if elasticity is not None:
            perm = (np.arange(dim)[:, None] + dim * np.arange(m.nv)[None, :]).ravel()   # blocked -> interleaved
            A = fo.assemble_elasticity(m, *elasticity)[perm][:, perm].tocsr()
        else:
            K, M = fo.assemble_stiffness_mass(m)
            A = (alpha * M + beta * K).tocsr()
        lv = Level()
        lv.n, lv.A, lv.ncomp = list(n), A, ncomp
        lv.mask = np.tile(dir_pred(m.coords, n), ncomp)
        lv.free = ~lv.mask
        d = A.diagonal()
        lv.dinv = np.where(lv.free, 1.0 / d, 0.0)
        lv.lmax = float(np.max(np.asarray(abs(A).sum(axis=1)).ravel() / d))
        F = sp.diags(lv.free.astype(float))
        lv.Am = (F @ A @ F).tocsr()
        if ncomp > 1:
            lv.lmax = power_lmax(lv)
        levels.append(lv)
        can = all(k % 2 == 0 and k >= 2 and k // 2 >= min_cells for k in n) and len(levels) < max_levels
        if can:
            nc = [k // 2 for k in n]
            mc = fo.make_mesh(dim, L, nc)
            if (~dir_pred(mc.coords, nc)).sum() == 0:
                can = False
        if not can:
            break
        n = [k // 2 for k in n]
    for a, b in zip(levels[:-1], levels[1:]):
        nf3 = a.n + [0] * (3 - dim)
        a.P = prolongation(nf3)
        if ncomp > 1:
            a.P = sp.kron(sp.identity(ncomp), a.P).tocsr()
    if lmax is not None:
        for lv, v in zip(levels, lmax):
            lv.lmax = float(v)
    lc = levels[-1]
    idx = np.nonzero(lc.free)[0]
    lc.dense = None
    # as Hierarchy::build: a dense inverse needs a small grid (nodes * ncomp <= 4 * 768) and at most 768 free dofs
    if len(levels) > 1 and lc.A.shape[0] <= 4 * dense_max and 0 < idx.size <= dense_max:
        lc.idx = idx
        lc.dense = np.linalg.inv(lc.Am[idx][:, idx].toarray())
    return levels


def cheby_coefs(lmax, ratio, sweeps):
    lmin = lmax / ratio
    theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    sigma = theta / delta
    rho = 1.0 / sigma
    out = [(0.0, 1.0 / theta)]
    for _ in range(1, sweeps):
        rn = 1.0 / (2 * sigma - rho)
        out.append((rn * rho, 2 * rn / delta))
        rho = rn
    return out


def smooth(lv, b, x, sweeps, ratio):
    d = np.zeros_like(b)
    for c1, c2 in cheby_coefs(lv.lmax, ratio, sweeps):
        r = lv.free * (b - lv.Am @ x)
        d = c1 * d + c2 * lv.dinv * r
        x = x + d
    return x


def vcycle(levels, b, nu=2, ratio=8.0, coarse_sweeps=8, l=0):
    lv = levels[l]
    if l == len(levels) - 1:
        if lv.dense is not None:
            x = np.zeros_like(b)
            x[lv.idx] = lv.dense @ b[lv.idx]
            return x
        return smooth(lv, b, np.zeros_like(b), nu if len(levels) == 1 else coarse_sweeps, ratio if len(levels) == 1 else 30.0)
    x = smooth(lv, b, np.zeros_like(b), nu, ratio)
    r = lv.free * (b - lv.Am @ x)
    nxt = levels[l + 1]
    bc = nxt.free * (lv.P.T @ r)
    xc = vcycle(levels, bc, nu, ratio, coarse_sweeps, l + 1)
    x = x + lv.free * (lv.P @ xc)
    return smooth(lv, b, x, nu, ratio)


def pcg(levels, b, rtol=1e-10, max_iters=200, nu=2, ratio=8.0, use_mg=True):
    lv = levels[0]
    b = lv.free * b
    x = np.zeros_like(b)
    r = b.copy()
    prec = (lambda v: vcycle(levels, v, nu, ratio)) if use_mg else (lambda v: lv.dinv * v)
    z = prec(r)
    p = z.copy()
    rho = r @ z
    bn = np.linalg.norm(b)
    hist = []
    for it in range(1, max_iters + 1):
        q = lv.Am @ p
        a = rho / (p @ q)
        x += a * p
        r -= a * q
        hist.append(np.linalg.norm(r) / bn)
        if hist[-1] <= rtol:
            break
        z = prec(r)
        rn = r @ z
        p = z + (rn / rho) * p
        rho = rn
    return x, hist
