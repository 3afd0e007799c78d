// Weighted (curvilinear-coordinate) heat tools: the reference's cylindrical / spherical solvers
// (fenics_mcp_server.py:769-1464) run the same P1 backward-Euler loop on Interval/Rectangle/Box meshes of the
// coordinate space with ONE scalar weight in every term,
//     a = w u v dx + dt k w grad(u).grad(v) dx ,   L = w u_n v dx + dt w f v dx ,
// w = x0 (degree 1), x0^2 or x0^2 sin(x1) (degree 2).  FFC interpolates a degree-p Expression into P_p on every
// cell and integrates exactly; the weight is separable, so its vertex / edge-midpoint values come from one table
// per axis on the half-step lattice.  The operator is no longer a constant stencil: k_wassemble writes the 15
// (7 / 3) stencil coefficients of every node once, k_vapply applies them, and a Jacobi-PCG with device-side
// scalars solves the systems.  Jacobi needs O(1/h) iterations, so precond = GMG switches to Galerkin multigrid
// (wmg.cu: symmetric half-coefficient storage, P^T A P coarse operators) when every axis halves evenly; the full
// stencil stays allocated for the true residual of that path.
//
// The cylinder / composite-core branches of _solve_heat_3d_raw (:512-572, 642-645) run through the same kernels: the
// reference's deployment has no mshr (neither Dockerfile nor requirements.txt install it), so its "cylinder" is
// BoxMesh((0,-R,-R),(Lx,R,R)) with every term weighted by Expression("sqrt(x[1]^2+x[2]^2)", degree=2)
// (weight_kind 1: not separable, evaluated from the y/z coordinate tables), and a composite core is a DG0
// diffusivity: core_diffusivity on the cells whose vertices and midpoint all have sqrt(y^2+z^2) < core_radius.
#include <chrono>
#include <cmath>
#include <cstring>
#include <memory>
#include <new>

#include "wmg.cuh"

struct WeightInts {
  int nk, nv;          // weight basis functions (P1: nv, P2: nv + edges), simplex vertices
  int ea[6], eb[6];    // edge (a,b) of weight basis function nv + e
  double Ws[10];       // int psi_k            (unit-volume simplex)
  double Wl[10][4];    // int psi_k lam_i
  double Wm[10][4][4]; // int psi_k lam_i lam_j
};

static double mono(int d, const int* ex, int n) {
  auto fac = [](int k) { double f = 1; for (int i = 2; i <= k; ++i) f *= i; return f; };
  double num = fac(d);
  int tot = 0;
  for (int i = 0; i < n; ++i) { num *= fac(ex[i]); tot += ex[i]; }
  return num / fac(d + tot);
}

static void build_weight_ints(int d, int degree, WeightInts* w) {
  std::memset(w, 0, sizeof(*w));
  const int nv = d + 1;
  w->nv = nv;
  struct Term { double cf; int ex[4]; };
  std::vector<std::vector<Term>> polys;
  for (int v = 0; v < nv; ++v) {
    std::vector<Term> p;
    if (degree == 1) { Term t{1.0, {0, 0, 0, 0}}; t.ex[v] = 1; p.push_back(t); }
    else {
      Term t2{2.0, {0, 0, 0, 0}}; t2.ex[v] = 2; p.push_back(t2);
      Term t1{-1.0, {0, 0, 0, 0}}; t1.ex[v] = 1; p.push_back(t1);
    }
    polys.push_back(p);
  }
  if (degree == 2) {
    int e = 0;
    for (int a = 0; a < nv; ++a)
      for (int b = a + 1; b < nv; ++b) {
        Term t{4.0, {0, 0, 0, 0}}; t.ex[a] += 1; t.ex[b] += 1;
        polys.push_back({t});
        w->ea[e] = a; w->eb[e] = b; ++e;
      }
  }
  w->nk = (int)polys.size();
  for (int k = 0; k < w->nk; ++k)
    for (const Term& t : polys[k]) {
      w->Ws[k] += t.cf * mono(d, t.ex, nv);
      for (int i = 0; i < nv; ++i) {
        int exi[4] = {t.ex[0], t.ex[1], t.ex[2], t.ex[3]};
        exi[i] += 1;
        w->Wl[k][i] += t.cf * mono(d, exi, nv);
        for (int j = 0; j < nv; ++j) {
          int exij[4] = {exi[0], exi[1], exi[2], exi[3]};
          exij[j] += 1;
          w->Wm[k][i][j] += t.cf * mono(d, exij, nv);
        }
      }
    }
}

// tab[m], m = ia + ib on the half-step lattice: weight factor of this axis at 0.5*(x[ia] + x[ib])
__global__ void __launch_bounds__(256)
k_weight_table(int dim, int n, double lo, double hi, int rpow, int use_sin, int len, double* __restrict__ tab) {
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < len; m += gridDim.x * blockDim.x) {
    const double ia = (double)(m / 2), ib = (double)((m + 1) / 2), dn = (double)n;
    const double L = __dsub_rn(hi, lo);
    double xa, xb;
    if (dim == 3) {  // BoxMesh: a + (i*(b-a))/n ; Interval/RectangleMesh: a + ((b-a)/n)*i
      xa = __dadd_rn(lo, __ddiv_rn(__dmul_rn(ia, L), dn));
      xb = __dadd_rn(lo, __ddiv_rn(__dmul_rn(ib, L), dn));
    } else {
      xa = __dadd_rn(lo, __dmul_rn(__ddiv_rn(L, dn), ia));
      xb = __dadd_rn(lo, __dmul_rn(__ddiv_rn(L, dn), ib));
    }
    const double x = 0.5 * (xa + xb);
    double v = 1.0;
    for (int p = 0; p < rpow; ++p) v *= x;
    if (use_sin) v *= sin(x);
    tab[m] = v;
  }
}

// per node: stencil rows of A = alpha*Mw + beta*Kw and of Mw, and the weighted load  m_i = int I(w) phi_i
__global__ void __launch_bounds__(128)
k_wassemble(const __grid_constant__ Grid g, const __grid_constant__ SimplexGeom sg, const __grid_constant__ WeightInts wi,
            double alpha, double beta, const double* __restrict__ tx, const double* __restrict__ ty,
            const double* __restrict__ tz, const double* __restrict__ cyt, const double* __restrict__ czt,
            int radial_yz, double core_radius, double beta_core,
            double* __restrict__ coefA, double* __restrict__ coefM, double* __restrict__ loadv) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const int gz = lz + g.z0;
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      double cA[PDE_NOFF], cM[PDE_NOFF], ld = 0.0;
#pragma unroll
      for (int k = 0; k < PDE_NOFF; ++k) cA[k] = cM[k] = 0.0;
      for (int o = 0; o < 8; ++o) {
        const int ox = o & 1, oy = (o >> 1) & 1, oz = (o >> 2) & 1;
        if ((ox && (g.nc[0] == 0 || ix == 0)) || (!ox && g.nc[0] > 0 && ix == g.nn[0] - 1)) continue;
        if ((oy && (g.nc[1] == 0 || iy == 0)) || (!oy && g.nc[1] > 0 && iy == g.nn[1] - 1)) continue;
        if ((oz && (g.nc[2] == 0 || gz == 0)) || (!oz && g.nc[2] > 0 && gz == g.nzg - 1)) continue;
        const int cx = ix - ox, cy = iy - oy, cz = gz - oz;  // corner 0 of the cell
        for (int t = 0; t < sg.nsimp; ++t) {
          int li = -1;
          for (int a = 0; a < sg.nv; ++a)
            if (sg.corner[t][a] == o) li = a;
          if (li < 0) continue;
          auto val = [&](int ca, int cb) {
            if (radial_yz) {  // w = sqrt(y^2 + z^2) at the vertex / edge midpoint
              const double yy = cyt[2 * cy + ((ca >> 1) & 1) + ((cb >> 1) & 1)];
              const double zz = czt[2 * cz + ((ca >> 2) & 1) + ((cb >> 2) & 1)];
              return sqrt(yy * yy + zz * zz);
            }
            double v = tx[2 * cx + (ca & 1) + (cb & 1)];
            if (g.nc[1] > 0) v *= ty[2 * cy + ((ca >> 1) & 1) + ((cb >> 1) & 1)];
            if (g.nc[2] > 0) v *= tz[2 * cz + ((ca >> 2) & 1) + ((cb >> 2) & 1)];
            return v;
          };
          double wk[10];
          for (int a = 0; a < sg.nv; ++a) wk[a] = val(sg.corner[t][a], sg.corner[t][a]);
          for (int e = 0; e < wi.nk - wi.nv; ++e) wk[wi.nv + e] = val(sg.corner[t][wi.ea[e]], sg.corner[t][wi.eb[e]]);
          double wbar = 0.0, wl = 0.0;
          for (int k = 0; k < wi.nk; ++k) { wbar = fma(wk[k], wi.Ws[k], wbar); wl = fma(wk[k], wi.Wl[k][li], wl); }
          double beta_t = beta;
          if (core_radius >= 0.0) {
            // SubDomain.mark (check_midpoint = true): every vertex and the cell midpoint inside r < core_radius
            bool inside = true;
            double my = 0.0, mz = 0.0;
            for (int a = 0; a < sg.nv; ++a) {
              const int ca = sg.corner[t][a];
              const double yy = cyt[2 * cy + 2 * ((ca >> 1) & 1)], zz = czt[2 * cz + 2 * ((ca >> 2) & 1)];
              inside = inside && (sqrt(yy * yy + zz * zz) < core_radius);
              my += yy; mz += zz;
            }
            my /= (double)sg.nv; mz /= (double)sg.nv;
            inside = inside && (sqrt(my * my + mz * mz) < core_radius);
            if (inside) beta_t = beta_core;
          }
          ld = fma(sg.vol, wl, ld);
          for (int b = 0; b < sg.nv; ++b) {
            const int cb = sg.corner[t][b];
            const int dx = (cb & 1) - ox, dy = ((cb >> 1) & 1) - oy, dz = ((cb >> 2) & 1) - oz;
            // index of the Kuhn offset (dx,dy,dz); the element split only produces offsets of that set
            int kk = 0;
            for (int k = 0; k < g.nk; ++k)
              if (g.kdx[k] == dx && g.kdy[k] == dy && g.kdz[k] == dz) kk = k;
            double gg = 0.0, wm = 0.0;
            for (int q = 0; q < 3; ++q) gg = fma(sg.G[t][li][q], sg.G[t][b][q], gg);
            for (int k = 0; k < wi.nk; ++k) wm = fma(wk[k], wi.Wm[k][li][b], wm);
            const double m = sg.vol * wm, kv = sg.vol * wbar * gg;
            cM[kk] += m;
            cA[kk] += alpha * m + beta_t * kv;
          }
        }
      }
      const long long idx = (long long)g.PX * iy + g.plane * lz + ix;
      for (int k = 0; k < g.nk; ++k) {
        coefA[idx + k * g.comp_stride] = cA[k];
        coefM[idx + k * g.comp_stride] = cM[k];
      }
      loadv[idx] = ld;
    }
  }
}

// y_i = by*y_i + a * sum_k coef_k[i] x[i+off_k] + gl * load_i on free rows, 0 on Dirichlet rows; sum x.y -> out
__global__ void __launch_bounds__(128)
k_vapply(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc, const double* __restrict__ coef,
         const double* __restrict__ x, double* __restrict__ y, const double* __restrict__ loadv, double by, double a,
         double gl, int do_reduce, ReduceBuf red, double* red_out) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  double acc_xy = 0.0, acc_yy = 0.0;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const long long rbase = (long long)g.PX * iy + g.plane * lz;
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const long long idx = rbase + ix;
      double bcv;
      if (bc_node(g, bc, ix, iy, lz + g.z0, &bcv)) { y[idx] = 0.0; continue; }
      double t = 0.0;
      for (int k = 0; k < g.nk; ++k) t = fma(coef[idx + k * g.comp_stride], x[idx + g.koff[k]], t);
      const double yv = (by != 0.0 ? by * y[idx] : 0.0) + a * t + (gl != 0.0 ? gl * loadv[idx] : 0.0);
      y[idx] = yv;
      acc_xy = fma(x[idx], yv, acc_xy);
      acc_yy = fma(yv, yv, acc_yy);
    }
  }
  if (do_reduce) {
    double v[2] = {acc_xy, acc_yy};
    block_reduce_finalize<2>(v, red, red_out);
  }
}

// Jacobi-PCG updates with the per-node diagonal coef_0:  x += a p, r -= a q, (r.D^-1 r, r.r) ;  p = D^-1 r + b p
__global__ void __launch_bounds__(128)
k_vcg_update(const __grid_constant__ Grid g, const double* __restrict__ diag, double* __restrict__ x,
             double* __restrict__ r, const double* __restrict__ p, const double* __restrict__ q,
             const double* __restrict__ scal, int s_rho, int s_pap, ReduceBuf red, double* out) {
  const double pap = scal[s_pap], rho = scal[s_rho];
  const double alpha = pap > 0.0 ? rho / pap : 0.0;
  const long long rows = (long long)g.nn[1] * g.nzl;
  double rz = 0.0, rr = 0.0;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const long long rbase = (long long)g.PX * (row % g.nn[1]) + g.plane * (row / g.nn[1]);
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const long long ii = rbase + ix;
      x[ii] = fma(alpha, p[ii], x[ii]);
      const double rv = fma(-alpha, q[ii], r[ii]);
      r[ii] = rv;
      const double d = diag[ii];
      rr = fma(rv, rv, rr);
      if (d > 0.0) rz = fma(rv / d, rv, rz);
    }
  }
  double v[2] = {rz, rr};
  block_reduce_finalize<2>(v, red, out);
}

__global__ void __launch_bounds__(128)
k_vcg_pupdate(const __grid_constant__ Grid g, const double* __restrict__ diag, double* __restrict__ p,
              const double* __restrict__ r, const double* __restrict__ scal, int s_rho, int s_rho_new, int first) {
  double beta = 0.0;
  if (!first) {
    const double rho = scal[s_rho];
    beta = rho > 0.0 ? scal[s_rho_new] / rho : 0.0;
  }
  const long long rows = (long long)g.nn[1] * g.nzl;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const long long rbase = (long long)g.PX * (row % g.nn[1]) + g.plane * (row / g.nn[1]);
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const long long ii = rbase + ix;
      const double d = diag[ii];
      const double z = d > 0.0 ? r[ii] / d : 0.0;
      p[ii] = first ? z : fma(beta, p[ii], z);
    }
  }
}

struct WheatState {
  pde_ctx* c;
  Grid g;
  BcDev bc;
  Field coefA, coefM, loadv, u, r, p, q;
  ~WheatState() {
    coefA.release(); coefM.release(); loadv.release(); u.release(); r.release(); p.release(); q.release();
  }
};

static int vapply(WheatState& s, const Field& coef, const double* x, double* y, double by, double a, double gl,
                  int slot) {
  pde_ctx* c = s.c;
  RowLaunch rl = row_launch(c, s.g);
  k_vapply<<<rl.grid, rl.block, 0, c->stream>>>(s.g, s.bc, coef.p, x, y, s.loadv.p, by, a, gl, slot >= 0, c->red,
                                                slot >= 0 ? c->scal + slot : nullptr);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// Jacobi-PCG on A x = b given x (with Dirichlet values) and r = masked(b - A x)
static int wpcg(WheatState& s, double bn2, const pde_solver_opts& o, pde_stats* st) {
  pde_ctx* c = s.c;
  const Grid& g = s.g;
  st->solves += 1;
  st->levels = 1;
  if (!(bn2 > 0.0)) { st->final_relres = 0.0; return 0; }
  const double tol2 = o.rtol * o.rtol * bn2;
  RowLaunch rl = row_launch(c, g);
  // rho0 = r.D^-1 r, rr0 (alpha = 0: slots S_XY hold 0)
  CUDA_OK(cudaMemsetAsync(c->scal + S_XY, 0, 2 * sizeof(double), c->stream));
  k_vcg_update<<<rl.grid, rl.block, 0, c->stream>>>(g, s.coefA.p, s.u.p, s.r.p, s.p.p, s.q.p, c->scal, S_RHO0, S_XY,
                                                    c->red, c->scal + S_RHO0);
  k_vcg_pupdate<<<rl.grid, rl.block, 0, c->stream>>>(g, s.coefA.p, s.p.p, s.r.p, c->scal, S_RHO0, S_RHO0, 1);
  c->launches += 2;
  double rr;
  PDE_OK(read_scal(c, S_RHO0 + 1, 1, &rr));
  int it = 0;
  bool conv = rr <= tol2;
  const int check = o.check_every > 0 ? o.check_every : 10;
  while (!conv && it < o.max_iters) {
    const int sr = 2 * (it & 1), sn = 2 * (1 - (it & 1));
    PDE_OK(vapply(s, s.coefA, s.p.p, s.q.p, 0.0, 1.0, 0.0, S_XY));   // q = A p, p.q
    k_vcg_update<<<rl.grid, rl.block, 0, c->stream>>>(g, s.coefA.p, s.u.p, s.r.p, s.p.p, s.q.p, c->scal, sr, S_XY,
                                                      c->red, c->scal + sn);
    k_vcg_pupdate<<<rl.grid, rl.block, 0, c->stream>>>(g, s.coefA.p, s.p.p, s.r.p, c->scal, sr, sn, 0);
    c->launches += 2;
    ++it;
    if (it % check == 0 || it >= o.max_iters) {
      PDE_OK(read_scal(c, sn + 1, 1, &rr));
      if (!(rr == rr)) PDE_FAIL("weighted PCG broke down (NaN residual)");
      conv = rr <= tol2;
    }
  }
  CUDA_OK(cudaGetLastError());
  st->iters_total += it;
  st->final_relres = std::sqrt(rr / bn2);
  if (!conv) st->converged = 0;
  return 0;
}

// validates p, lays out the grid (L: user box lengths) and assembles coefA / coefM / loadv into s
static int wheat_assemble(pde_ctx* c, const pde_wheat_params* p, WheatState& s, double L[3]) {
  if (c->world > 1) PDE_FAIL("pde_wheat_solve: the curvilinear tools run on one GPU");
  CUDA_OK(cudaSetDevice(c->device));
  if (p->dim < 1 || p->dim > 3) PDE_FAIL("dim must be 1, 2 or 3");
  if (p->weight_degree != 1 && p->weight_degree != 2) PDE_FAIL("weight_degree must be 1 or 2");
  if (p->weight_rpow < 0 || p->weight_rpow > 2) PDE_FAIL("weight_rpow must be 0, 1 or 2");
  if (p->weight_kind != 0 && p->weight_kind != 1) PDE_FAIL("weight_kind must be 0 (separable) or 1 (radial y-z)");
  if ((p->weight_kind == 1 || p->has_core) && p->dim != 3) PDE_FAIL("radial y-z weight / composite core need dim 3");
  if (p->has_core && !(p->core_diffusivity > 0)) PDE_FAIL("core_diffusivity must be > 0");
  if (!p->steady && !(p->dt > 0)) PDE_FAIL("dt must be > 0");
  if (!(p->diffusivity > 0)) PDE_FAIL("diffusivity must be > 0");
  for (int k = 0; k < 3; ++k) L[k] = 1.0;
  for (int k = 0; k < p->dim; ++k) {
    L[k] = p->hi[k] - p->lo[k];
    if (!(L[k] > 0)) PDE_FAIL("hi must exceed lo on every axis");
  }
  s.c = c;
  PDE_OK(make_grid(p->dim, p->n, L, 0, 1, &s.g));
  user_bc_to_dev(p->dim, &p->bc, &s.bc);
  const Grid& g = s.g;
  PDE_OK(s.coefA.alloc(c, g, PDE_NOFF));
  PDE_OK(s.coefM.alloc(c, g, PDE_NOFF));
  PDE_OK(s.loadv.alloc(c, g, 1));
  PDE_OK(s.u.alloc(c, g, 1));
  PDE_OK(s.r.alloc(c, g, 1));
  PDE_OK(s.p.alloc(c, g, 1));
  PDE_OK(s.q.alloc(c, g, 1));
  // weight tables on the half-step lattice, one per user axis (dim 2: user y is internal z)
  double* tabs[3] = {nullptr, nullptr, nullptr};
  struct TabRel { double** t; ~TabRel() { for (int q = 0; q < 3; ++q) if (t[q]) cudaFree(t[q]); } } tabrel{tabs};
  for (int q = 0; q < p->dim; ++q) {
    const int iax = (p->dim == 2 && q == 1) ? 2 : q;
    const int len = 2 * p->n[q] + 1;
    CUDA_OK(cudaMalloc(&tabs[iax], sizeof(double) * len));
    k_weight_table<<<(len + 255) / 256, 256, 0, c->stream>>>(p->dim, p->n[q], p->lo[q], p->hi[q],
                                                             q == 0 ? p->weight_rpow : 0, q == 1 ? p->weight_sin_axis1 : 0,
                                                             len, tabs[iax]);
    c->launches++;
  }
  // y / z coordinate tables on the half-step lattice (radial weight, core marking)
  double* ctabs[2] = {nullptr, nullptr};
  struct CTabRel { double** t; ~CTabRel() { for (int q = 0; q < 2; ++q) if (t[q]) cudaFree(t[q]); } } ctabrel{ctabs};
  if (p->weight_kind == 1 || p->has_core)
    for (int q = 1; q < 3; ++q) {
      const int len = 2 * p->n[q] + 1;
      CUDA_OK(cudaMalloc(&ctabs[q - 1], sizeof(double) * len));
      k_weight_table<<<(len + 255) / 256, 256, 0, c->stream>>>(3, p->n[q], p->lo[q], p->hi[q], 1, 0, len, ctabs[q - 1]);
      c->launches++;
    }
  SimplexGeom sg;
  build_simplex_geom(p->dim, g.h, &sg);
  WeightInts wi;
  build_weight_ints(p->dim, p->weight_degree, &wi);
  const double kappa = p->diffusivity;
  const double alpha = p->steady ? 0.0 : 1.0, beta = p->steady ? kappa : p->dt * kappa;
  RowLaunch rl = row_launch(c, g);
  k_wassemble<<<rl.grid, rl.block, 0, c->stream>>>(g, sg, wi, alpha, beta, tabs[0], tabs[1] ? tabs[1] : tabs[0],
                                                   tabs[2] ? tabs[2] : tabs[0], ctabs[0], ctabs[1], p->weight_kind == 1,
                                                   p->has_core ? p->core_radius : -1.0,
                                                   p->steady ? p->core_diffusivity : p->dt * p->core_diffusivity,
                                                   s.coefA.p, s.coefM.p, s.loadv.p);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// Resident stepper: the assembled operator, the multigrid hierarchy and the field stay on the device between calls.
// pde_wheat_solve runs on the same pieces (wheat_setup, wheat_init_state, wheat_advance, wheat_get_state).
struct pde_wheat_state : WheatState {
  pde_wheat_params prm{};
  pde_solver_opts o{};
  double L[3] = {1.0, 1.0, 1.0};
  WHierarchy mg;
  bool use_mg = false;
  double setup_ms = 0.0;   // host time of the hierarchy set-up
  Field un;                // u_n of a verified step (true residual), allocated on first use
  double* dense = nullptr; // [nloc] natural-order staging buffer of the host copies
  long long nloc = 0;
  ~pde_wheat_state() {
    un.release();
    if (dense) cudaFree(dense);
  }
};

// everything before the initial state: checks, assembly, the GMG hierarchy (PDE_PRECOND_AUTO keeps Jacobi here; a
// grid that does not coarsen runs Jacobi), the staging buffer
static int wheat_setup(pde_ctx* c, const pde_wheat_params* p, const pde_solver_opts* o_in, pde_wheat_state* s) {
  if (p->initial_type == PDE_IC_ARRAY) PDE_FAIL("initial_type array: load the field with pde_wheat_set_state");
  s->prm = *p;
  if (o_in) s->o = *o_in; else pde_solver_opts_default(&s->o);
  PDE_OK(wheat_assemble(c, p, *s, s->L));
  if (s->o.precond == PDE_PRECOND_GMG) {
    CUDA_OK(cudaStreamSynchronize(c->stream));
    const auto t0 = std::chrono::steady_clock::now();
    PDE_OK(s->mg.build(c, s->g, s->bc, s->coefA.p));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    s->setup_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    s->use_mg = s->mg.levels() >= 2;
    if (!s->use_mg) s->mg.release();
  }
  s->nloc = (long long)s->g.nn[0] * s->g.nn[1] * s->g.nzg;
  CUDA_OK(cudaMalloc(&s->dense, sizeof(double) * s->nloc));
  return 0;
}

// initial state / Dirichlet lift: every initial_type of the curvilinear tools falls back to the constant
// (:893-896 ...); the 3D cylinder / composite branches keep zero and the (unweighted) cosine / sine projection
static int wheat_init_state(pde_wheat_state& s) {
  const pde_wheat_params& p = s.prm;
  if (!p.steady && (p.initial_type == PDE_IC_COSINE || p.initial_type == PDE_IC_SINE)) {
    PDE_OK(project_trig_ic(s.c, s.g, s.bc, p.dim, p.n, s.L, p.lo, p.initial_amplitude, p.initial_wavenumber,
                           p.initial_type == PDE_IC_SINE, s.o, s.u.p, s.r.p));
  } else {
    const double v0 = (p.steady || p.initial_type == PDE_IC_ZERO) ? 0.0 : p.T_initial;
    PDE_OK(launch_fill_ic(s.c, s.g, s.bc, s.u.p, v0, 1));
  }
  return 0;
}

static void wheat_stats(const pde_wheat_state& s, pde_stats* st) {
  std::memset(st, 0, sizeof(*st));
  st->ndofs = s.nloc;
  st->converged = 1;
  st->true_relres = NAN;
  st->setup_ms = s.setup_ms;
}

// nsteps backward-Euler steps (steady: the one solve, u is the starting guess), accumulated into st.  verify_last: on
// the GMG path (verify_residual >= 0), ||b - A x|| / ||b|| of the last step with the full assembled stencil (this also
// checks the packed operator)
static int wheat_advance(pde_wheat_state& s, int nsteps, bool verify_last, pde_stats* st) {
  pde_ctx* c = s.c;
  const Grid& g = s.g;
  const pde_wheat_params& p = s.prm;
  const double f = p.source_value;
  const bool verify = verify_last && s.use_mg && s.o.verify_residual >= 0;
  auto solve = [&](double bn2) -> int {
    return s.use_mg ? wmg_pcg(c, s.mg, s.u.p, s.r.p, s.p.p, s.q.p, bn2, s.o, st) : wpcg(s, bn2, s.o, st);
  };
  if (p.steady) {
    if (nsteps < 1) return 0;
    // r0 = f m_w - k K_w u  (A = k K_w)
    PDE_OK(vapply(s, s.coefA, s.u.p, s.r.p, 0.0, -1.0, f, S_XY));
    double bn2;
    PDE_OK(read_scal(c, S_YY, 1, &bn2));
    PDE_OK(solve(bn2));
    if (verify) {
      PDE_OK(vapply(s, s.coefA, s.u.p, s.q.p, 0.0, -1.0, f, S_XY));
      double rr;
      PDE_OK(read_scal(c, S_YY, 1, &rr));
      st->true_relres = bn2 > 0 ? std::sqrt(rr / bn2) : 0.0;
    }
    return 0;
  }
  for (int step = 0; step < nsteps; ++step) {
    const bool last = verify && step == nsteps - 1;
    if (last) {
      if (!s.un.p) PDE_OK(s.un.alloc(c, g, 1));
      PDE_OK(launch_copy(c, g, 1, s.un.p, s.u.p));
    }
    // b = M_w u_n + dt f m_w (its norm is the stopping scale); warm start x0 = u_n: r0 = b - A u_n
    PDE_OK(vapply(s, s.coefM, s.u.p, s.r.p, 0.0, 1.0, p.dt * f, S_XY));
    double bn2;
    PDE_OK(read_scal(c, S_YY, 1, &bn2));
    PDE_OK(vapply(s, s.coefA, s.u.p, s.r.p, 1.0, -1.0, 0.0, -1));
    PDE_OK(solve(bn2));
    if (last) {
      PDE_OK(vapply(s, s.coefM, s.un.p, s.q.p, 0.0, 1.0, p.dt * f, -1));
      PDE_OK(vapply(s, s.coefA, s.u.p, s.q.p, 1.0, -1.0, 0.0, S_XY));
      double rr;
      PDE_OK(read_scal(c, S_YY, 1, &rr));
      st->true_relres = bn2 > 0 ? std::sqrt(rr / bn2) : 0.0;
    }
  }
  return 0;
}

static int wheat_get_state(pde_wheat_state& s, double* dst) {
  PDE_OK(launch_pack(s.c, s.g, 1, s.u.p, s.dense, 0));
  return d2h(s.c, dst, s.dense, sizeof(double) * s.nloc);
}

extern "C" int pde_wheat_close(pde_wheat_state* s) {
  if (!s) return 0;
  cudaSetDevice(s->c->device);
  cudaStreamSynchronize(s->c->stream);
  delete s;
  return 0;
}

extern "C" int pde_wheat_open(pde_ctx* c, const pde_wheat_params* p, const pde_solver_opts* o, pde_wheat_state** out) {
  if (!c || !p || !out) PDE_FAIL("null argument");
  pde_wheat_state* s = new (std::nothrow) pde_wheat_state();
  if (!s) PDE_FAIL("out of host memory");
  s->c = c;
  int rc = wheat_setup(c, p, o, s);
  if (!rc) rc = wheat_init_state(*s);
  if (rc) {
    pde_wheat_close(s);
    return rc;
  }
  *out = s;
  return 0;
}

extern "C" int64_t pde_wheat_local_nverts(pde_wheat_state* s) { return s ? s->nloc : 0; }

extern "C" int pde_wheat_set_state(pde_wheat_state* s, const double* u_host) {
  if (!s || !u_host) PDE_FAIL("null argument");
  pde_ctx* c = s->c;
  CUDA_OK(cudaSetDevice(c->device));
  PDE_OK(h2d(c, s->dense, u_host, sizeof(double) * s->nloc));
  PDE_OK(launch_unpack(c, s->g, 1, s->dense, s->u.p, 0));
  return launch_apply_bc_values(c, s->g, s->bc, s->u.p);
}

extern "C" int pde_wheat_get_state(pde_wheat_state* s, double* u_host) {
  if (!s || !u_host) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(s->c->device));
  return wheat_get_state(*s, u_host);
}

extern "C" int pde_wheat_step(pde_wheat_state* s, int nsteps, pde_stats* st_out) {
  if (!s) PDE_FAIL("null state");
  if (nsteps < 0) PDE_FAIL("nsteps must be >= 0");
  pde_ctx* c = s->c;
  CUDA_OK(cudaSetDevice(c->device));
  pde_stats st;
  wheat_stats(*s, &st);
  const long long l0 = c->launches;
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  PDE_OK(wheat_advance(*s, nsteps, true, &st));
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  st.solve_ms = ms;
  st.launches = c->launches - l0;
  if (st_out) *st_out = st;
  return 0;
}

// open, step(1) per step with a snapshot every snapshot_stride steps, close.  solve_ms is the device time from the
// initial state to the last snapshot; the set-up (assembly, hierarchy) is not part of it.
extern "C" int pde_wheat_solve(pde_ctx* c, const pde_wheat_params* p, const pde_solver_opts* o, double* values_out,
                               double* times_out, pde_stats* st_out) {
  if (!c || !p || !values_out || !times_out) PDE_FAIL("null argument");
  std::unique_ptr<pde_wheat_state> s(new (std::nothrow) pde_wheat_state());
  if (!s) PDE_FAIL("out of host memory");
  s->c = c;
  PDE_OK(wheat_setup(c, p, o, s.get()));
  pde_stats st;
  wheat_stats(*s, &st);
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  const long long l0 = c->launches;
  PDE_OK(wheat_init_state(*s));
  if (p->steady) {
    PDE_OK(wheat_advance(*s, 1, true, &st));
    PDE_OK(wheat_get_state(*s, values_out));
    times_out[0] = 0.0;
  } else {
    long long snap = 0;
    PDE_OK(wheat_get_state(*s, values_out));
    times_out[snap++] = 0.0;
    const int stride = p->snapshot_stride > 0 ? p->snapshot_stride : 1;
    for (int step = 0; step < p->num_steps; ++step) {
      PDE_OK(wheat_advance(*s, 1, step == p->num_steps - 1, &st));
      if ((step + 1) % stride == 0) {
        PDE_OK(wheat_get_state(*s, values_out + snap * s->nloc));
        times_out[snap++] = (step + 1) * p->dt;
      }
    }
  }
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  st.solve_ms = ms;
  st.launches = c->launches - l0;
  if (st_out) *st_out = st;
  return 0;
}

extern "C" int pde_wheat_level_coefs(pde_ctx* c, const pde_wheat_params* p, int level, int32_t n_out[3],
                                     double* coef_out) {
  if (!c || !p || !n_out) PDE_FAIL("null argument");
  WheatState s;
  double L[3];
  PDE_OK(wheat_assemble(c, p, s, L));
  WHierarchy mg;
  PDE_OK(mg.build(c, s.g, s.bc, s.coefA.p));
  if (level < 0 || level >= mg.levels()) PDE_FAIL("no such multigrid level");
  for (int q = 0; q < 3; ++q) n_out[q] = q < p->dim ? p->n[q] >> level : 0;
  if (coef_out) PDE_OK(wmg_level_coefs(c, mg, level, coef_out));
  return 0;
}

// Test entry: the V-cycle of pde_wheat_solve's GMG path applied ncycles times to one host vector (see the header)
extern "C" int pde_wheat_vcycle(pde_ctx* c, const pde_wheat_params* p, int32_t ncycles, const double* b, double* z_first,
                                double* z_last, double* bz, pde_mg_info* info) {
  if (!c || !p || !b || !z_first || !z_last || !info) PDE_FAIL("null argument");
  if (ncycles < 1) PDE_FAIL("ncycles must be >= 1");
  WheatState s;
  double L[3];
  PDE_OK(wheat_assemble(c, p, s, L));
  WHierarchy mg;
  PDE_OK(mg.build(c, s.g, s.bc, s.coefA.p));
  const int nl = mg.levels();
  if (nl < 2) PDE_FAIL("weighted multigrid: the grid does not coarsen");
  if (nl > PDE_MG_MAX_LEVELS) PDE_FAIL("more multigrid levels than pde_mg_info holds");
  const Grid& g = s.g;
  const size_t bytes = sizeof(double) * g.nn[0] * g.nn[1] * g.nzg;
  double* dense = nullptr;
  CUDA_OK(cudaMalloc(&dense, bytes));
  struct DenseRel { double* p; ~DenseRel() { cudaFree(p); } } denserel{dense};
  PDE_OK(h2d(c, dense, b, bytes));
  PDE_OK(launch_unpack(c, g, 1, dense, s.r.p, 0));
  for (int k = 0; k < ncycles; ++k) {
    double* z = nullptr;
    PDE_OK(wvcycle(c, mg, s.r.p, &z, S_RHO0));
    if (k == 0 || k == ncycles - 1) PDE_OK(launch_pack(c, g, 1, z, dense, 0));
    if (k == 0) PDE_OK(d2h(c, z_first, dense, bytes));
    if (k == ncycles - 1) PDE_OK(d2h(c, z_last, dense, bytes));
  }
  if (bz) PDE_OK(read_scal(c, S_RHO0, 1, bz));
  std::memset(info, 0, sizeof(*info));
  info->levels = nl;
  info->n_dense = mg.lv[nl - 1]->n_dense;
  int ax[3], nax;
  internal_axes(p->dim, ax, &nax);
  for (int l = 0; l < nl; ++l) {
    for (int q = 0; q < nax; ++q) info->n[l][q] = mg.lv[l]->g.nc[ax[q]];
    info->lmax[l] = mg.lv[l]->lmax;
  }
  return 0;
}
