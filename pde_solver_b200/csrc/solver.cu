// Operators, geometric multigrid hierarchy and the PCG driver.
//
// Replaces the linear-algebra half of the reference's `solve(a == L, u, bcs)` calls
// (fenics_mcp_server.py:265,311,397,440,661,709,1538,1688,1838: assemble AIJ + sparse LU every call)
// with a matrix-free preconditioned CG whose operator is never stored.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "solver.cuh"

int launch_stencil_generic(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a);
int launch_stencil_fast(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a, bool* handled);
int launch_heat_post2(pde_ctx* c, const Grid& g, const OpDev& op, const double* x0, const double* b, double* y, double c2_0,
                      double c1_1, double c2_1, int dot_slot, bool* handled);
bool elast3d_first2_ok(const Grid& g, const BcDev& bc, const OpDev& op);
bool post2_applicable(const Grid& g, const OpDev& op);
int launch_heat_resid_restrict(pde_ctx* c, const Grid& gf, const Grid& gc, const OpDev& op, const double* x, const double* b,
                               double* bcoarse, bool* handled);

int launch_stencil(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a) {
  if (a.variant == 0) {
    bool handled = false;
    PDE_OK(launch_stencil_fast(c, g, bc, op, a, &handled));
    if (handled) return 0;
  }
  return launch_stencil_generic(c, g, bc, op, a);
}

// ---- Field ---------------------------------------------------------------------------------
int Field::alloc(pde_ctx* c, const Grid& g, int ncomp) {
  release();
  // lead/tail pad: the (-1,-1,-1) neighbour of node (0,0,0) lies PX+1 elements before the ghost plane
  const size_t lead = (((size_t)g.PX + 1 + 31) / 32) * 32;
  bytes = ((size_t)g.comp_stride * ncomp + 2 * lead) * sizeof(double);
  CUDA_OK(cudaMalloc(&raw, bytes));
  // zero on the context's stream: it is a non-blocking stream, so a legacy-stream cudaMemset would
  // not be ordered against the kernels that use this field
  CUDA_OK(cudaMemsetAsync(raw, 0, bytes, c->stream));
  p = raw + lead + PDE_NG * g.plane;
  return 0;
}
void Field::release() {
  if (raw) cudaFree(raw);
  raw = p = nullptr;
  bytes = 0;
}

// ---- Operator --------------------------------------------------------------------------------
int Operator::upload(pde_ctx* c) {
  const int nc = tab.ncomp, nn = nc * nc;
  dev.ncomp = nc;
  dev.gershgorin = tab.gershgorin;
  std::vector<double> dinv((size_t)PDE_NCLASS * nc, 0.0);
  for (int cls = 0; cls < PDE_NCLASS; ++cls)
    for (int i = 0; i < nc; ++i) {
      double dg = tab.coef[((size_t)cls * PDE_NOFF + 0) * nn + i * nc + i];
      dinv[cls * nc + i] = dg > 0 ? 1.0 / dg : 0.0;
    }
  for (int k = 0; k < PDE_NOFF; ++k)
    for (int q = 0; q < nn; ++q) dev.h_int[k * nn + q] = tab.coef[((size_t)13 * PDE_NOFF + k) * nn + q];
  for (int i = 0; i < nc; ++i) dev.h_dinv_int[i] = dinv[13 * nc + i];
  dev.h_load_int = tab.load[13];
  {
    // all faces of the present axes Dirichlet (and no other_faces exclusion): every free node is interior class
    bool u = !bc.side_excl;
    for (int ax = 0; ax < 3; ++ax)
      if (g.nc[ax] > 0 && !(bc.on[2 * ax] && bc.on[2 * ax + 1])) u = false;
    dev.uniform_diag = u ? 1 : 0;
  }
  CUDA_OK(cudaMalloc(&dev.coef, tab.coef.size() * sizeof(double)));
  CUDA_OK(cudaMalloc(&dev.dinv, dinv.size() * sizeof(double)));
  CUDA_OK(cudaMalloc(&dev.load, PDE_NCLASS * sizeof(double)));
  CUDA_OK(cudaMemcpyAsync(dev.coef, tab.coef.data(), tab.coef.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(cudaMemcpyAsync(dev.dinv, dinv.data(), dinv.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(cudaMemcpyAsync(dev.load, tab.load.data(), PDE_NCLASS * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(cudaStreamSynchronize(c->stream));  // host staging vectors die at return
  return 0;
}
int Operator::setup_scalar(pde_ctx* c, const Grid& g_, const BcDev& bc_, double alpha, double beta) {
  release();
  g = g_;
  bc = bc_;
  PDE_OK(build_scalar_table(g.dim, g.h, g.nc, alpha, beta, &tab));
  return upload(c);
}
int Operator::setup_elasticity(pde_ctx* c, const Grid& g_, const BcDev& bc_, double lam, double mu) {
  release();
  g = g_;
  bc = bc_;
  PDE_OK(build_elasticity_table(g.dim, g.h, g.nc, lam, mu, &tab));
  return upload(c);
}
void Operator::release() {
  if (dev.coef) cudaFree(dev.coef);
  if (dev.dinv) cudaFree(dev.dinv);
  if (dev.load) cudaFree(dev.load);
  dev.coef = dev.dinv = dev.load = nullptr;
}

// Scalars reach the host through mapped pinned memory written by a one-warp kernel, not through a copy engine: a
// cudaMemcpyAsync poll would queue behind the GB-sized snapshot transfers that run on the copy streams
// (pde_heat_advance_batch) and stall every convergence check for the length of a transfer.
__global__ void k_publish_scal(const double* __restrict__ src, double* __restrict__ dst_host, int count) {
  if ((int)threadIdx.x < count) dst_host[threadIdx.x] = src[threadIdx.x];
  __threadfence_system();
}

int read_scal(pde_ctx* c, int slot, int count, double* out) {
  if (count > 32) PDE_FAIL("read_scal: at most 32 slots per call");
  if (!c->h_scal_dev) CUDA_OK(cudaHostGetDevicePointer((void**)&c->h_scal_dev, c->h_scal, 0));
  k_publish_scal<<<1, 32, 0, c->stream>>>(c->scal + slot, c->h_scal_dev + slot, count);
  c->launches++;
  CUDA_OK(cudaStreamSynchronize(c->stream));
  if (c->world > 1) PDE_OK(comm_check_error(c));
  for (int i = 0; i < count; ++i) out[i] = ((volatile double*)c->h_scal)[slot + i];
  return 0;
}

// u = project(Expression("A cos(k x0) cos(k x1) ...", degree=2), V), then bc.apply(u) (reference :276-290, 408-421,
// 672-685): consistent-mass Jacobi-PCG (rtol 1e-13) of the exactly integrated P2-interpolated expression.  `rhs` is
// scratch; lo_user shifts the box (nullptr: box at the origin).
int project_trig_ic(pde_ctx* c, const Grid& g, const BcDev& bc, int dim, const int32_t n_user[3], const double L_user[3],
                    const double* lo_user, double amp, double kw, int use_sin, const pde_solver_opts& o, double* u,
                    double* rhs) {
  BcDev nobc;
  std::memset(&nobc, 0, sizeof(nobc));
  Operator Mf;
  PcgWork pw;
  int rc = 0;
  do {
    if ((rc = Mf.setup_scalar(c, g, nobc, 1.0, 0.0))) break;
    SimplexGeom sg;
    build_simplex_geom(dim, g.h, &sg);
    if ((rc = launch_p2_load(c, g, sg, amp, kw, use_sin, n_user, L_user, rhs, lo_user))) break;
    if ((rc = launch_zero(c, g, 1, u))) break;
    if ((rc = launch_dot(c, g, 1, rhs, rhs, S_TMP0))) break;
    if (c->world > 1 && (rc = comm_allreduce_scal(c, S_TMP0, 1))) break;
    double bn2;
    if ((rc = read_scal(c, S_TMP0, 1, &bn2))) break;
    if ((rc = pw.alloc(c, g, 1))) break;
    pde_solver_opts po = o;
    po.precond = PDE_PRECOND_JACOBI;
    po.rtol = 1e-13;
    pde_stats pst;
    std::memset(&pst, 0, sizeof(pst));
    pst.converged = 1;
    if ((rc = pcg_solve(c, Mf, nullptr, pw, u, rhs, bn2, po, &pst))) break;
    if (!pst.converged) { pde_set_error("initial-condition projection did not converge"); rc = 1; break; }
    if ((rc = launch_apply_bc_values(c, g, bc, u))) break;
  } while (0);
  cudaStreamSynchronize(c->stream);
  Mf.release();
  pw.release();
  return rc;
}

// ---- multigrid ---------------------------------------------------------------------------------
long long count_free_and_index(const Grid& g, const BcDev& bc, int ncomp, std::vector<long long>* idx,
                                      std::vector<int>* dofid) {
  long long n = 0;
  if (dofid) dofid->assign((size_t)g.nn[0] * g.nn[1] * g.nzl * ncomp, -1);
  for (int lz = 0; lz < g.nzl; ++lz)
    for (int iy = 0; iy < g.nn[1]; ++iy)
      for (int ix = 0; ix < g.nn[0]; ++ix) {
        double v;
        if (bc_node(g, bc, ix, iy, lz + g.z0, &v)) continue;
        for (int i = 0; i < ncomp; ++i) {
          if (idx) idx->push_back((long long)ix + (long long)g.PX * iy + g.plane * lz + i * g.comp_stride);
          if (dofid) (*dofid)[(((size_t)lz * g.nn[1] + iy) * g.nn[0] + ix) * ncomp + i] = (int)n;
          ++n;
        }
      }
  return n;
}

int dense_inverse_spd(std::vector<double>& A, int n) {
  // Cholesky A = L L^T (in place, lower), then A^-1 = L^-T L^-1
  for (int j = 0; j < n; ++j) {
    double d = A[(size_t)j * n + j];
    for (int k = 0; k < j; ++k) d -= A[(size_t)j * n + k] * A[(size_t)j * n + k];
    if (!(d > 0)) return 1;
    d = std::sqrt(d);
    A[(size_t)j * n + j] = d;
    for (int i = j + 1; i < n; ++i) {
      double s = A[(size_t)i * n + j];
      for (int k = 0; k < j; ++k) s -= A[(size_t)i * n + k] * A[(size_t)j * n + k];
      A[(size_t)i * n + j] = s / d;
    }
  }
  std::vector<double> Li((size_t)n * n, 0.0);
  for (int j = 0; j < n; ++j) {
    Li[(size_t)j * n + j] = 1.0 / A[(size_t)j * n + j];
    for (int i = j + 1; i < n; ++i) {
      double s = 0;
      for (int k = j; k < i; ++k) s -= A[(size_t)i * n + k] * Li[(size_t)k * n + j];
      Li[(size_t)i * n + j] = s / A[(size_t)i * n + i];
    }
  }
  for (int i = 0; i < n; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = 0;
      for (int k = i; k < n; ++k) s += Li[(size_t)k * n + i] * Li[(size_t)k * n + j];
      A[(size_t)i * n + j] = A[(size_t)j * n + i] = s;
    }
  return 0;
}

// Dense inverse of the coarsest operator.  It is built on the GLOBAL coarse grid (identical on every
// rank); idx maps global free dof j to this rank's flat local index, or -1 if another rank owns it.
static int build_dense_coarse(pde_ctx* c, MGLevel& L, int dim, const int32_t n_user[3], const double L_user[3]) {
  const Grid& gl = L.op.g;
  const int nc = L.op.tab.ncomp, nn = nc * nc;
  Grid g;  // global view
  PDE_OK(make_grid(dim, n_user, L_user, 0, 1, &g));
  std::vector<long long> idx;
  std::vector<int> dofid;
  long long n = count_free_and_index(g, L.op.bc, nc, &idx, &dofid);
  std::vector<double> A((size_t)n * n, 0.0);
  for (int lz = 0; lz < g.nzl; ++lz)
    for (int iy = 0; iy < g.nn[1]; ++iy)
      for (int ix = 0; ix < g.nn[0]; ++ix) {
        const size_t node = ((size_t)lz * g.nn[1] + iy) * g.nn[0] + ix;
        if (dofid[node * nc] < 0) continue;
        const int cls = node_class(g, ix, iy, lz + g.z0);
        for (int k = 0; k < g.nk; ++k) {
          int jx = ix + g.kdx[k], jy = iy + g.kdy[k], jz = lz + g.kdz[k];
          if (jx < 0 || jx >= g.nn[0] || jy < 0 || jy >= g.nn[1] || jz < 0 || jz >= g.nzl) continue;
          const size_t nb = ((size_t)jz * g.nn[1] + jy) * g.nn[0] + jx;
          if (dofid[nb * nc] < 0) continue;
          const double* cf = &L.op.tab.coef[((size_t)cls * PDE_NOFF + g.kidx[k]) * nn];
          for (int i = 0; i < nc; ++i)
            for (int j = 0; j < nc; ++j) A[(size_t)dofid[node * nc + i] * n + dofid[nb * nc + j]] += cf[i * nc + j];
        }
      }
  if (dense_inverse_spd(A, (int)n)) PDE_FAIL("coarse operator is not positive definite");
  // global flat index -> local flat index (or -1)
  for (auto& v : idx) {
    const int comp = (int)(v / g.comp_stride);
    const long long r = v % g.comp_stride;
    const int gz = (int)(r / g.plane);
    const long long inplane = r % g.plane;
    if (gz < gl.z0 || gz >= gl.z0 + gl.nzl) v = -1;
    else v = inplane + gl.plane * (gz - gl.z0) + comp * gl.comp_stride;
  }
  L.n_dense = (int)n;
  CUDA_OK(cudaMalloc(&L.Ainv, A.size() * sizeof(double)));
  CUDA_OK(cudaMalloc(&L.idx, idx.size() * sizeof(long long)));
  CUDA_OK(cudaMalloc(&L.bglob, (size_t)n * sizeof(double)));
  CUDA_OK(cudaMemcpyAsync(L.Ainv, A.data(), A.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(cudaMemcpyAsync(L.idx, idx.data(), idx.size() * sizeof(long long), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

// lmax(D^-1 A) of a level by power iteration (vector operators only: Gershgorin is tight for the scalar
// stencils but ~1.5x too large for the elasticity blocks, which weakens the Chebyshev smoother).
// Result: min(Gershgorin bound, 1.1 * power estimate); identical on every rank (all-reduced dots).
static int estimate_lmax(pde_ctx* c, MGLevel& L, int iters) {
  const Grid& g = L.op.g;
  const int nc = L.op.dev.ncomp;
  double* x = L.xa.p;
  double* y = L.xb.p;
  // deterministic start vector with all frequencies: x_i = sin(0.37 i) + 0.5 on free nodes
  PDE_OK(launch_fill_pattern(c, g, L.op.bc, nc, x));
  double lam = 0.0;
  for (int it = 0; it < iters; ++it) {
    StencilArgs a;
    a.x = x; a.y = y; a.reduce_slot_xy = S_TMP0;
    if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, x));
    PDE_OK(launch_stencil(c, g, L.op.bc, L.op.dev, a));
    PDE_OK(launch_cheby_first(c, g, L.op.bc, L.op.dev, y, y, 1.0));  // y <- D^-1 y
    PDE_OK(launch_dot(c, g, nc, y, y, S_TMP0));
    PDE_OK(launch_dot(c, g, nc, x, x, S_TMP1));
    if (c->world > 1 && !L.replicated) PDE_OK(comm_allreduce_scal(c, S_TMP0, 2));
    double v[2];
    PDE_OK(read_scal(c, S_TMP0, 2, v));
    if (!(v[1] > 0.0) || !(v[0] > 0.0)) break;
    lam = std::sqrt(v[0] / v[1]);
    // x <- y / ||y||
    PDE_OK(launch_zero(c, g, nc, x));
    PDE_OK(launch_axpy(c, g, nc, x, y, 1.0 / std::sqrt(v[0])));
  }
  PDE_OK(launch_zero(c, g, nc, L.xa.p));
  PDE_OK(launch_zero(c, g, nc, L.xb.p));
  PDE_OK(launch_zero(c, g, nc, L.r.p));
  if (lam > 0.0) {
    const double est = 1.1 * lam;
    if (est < L.op.dev.gershgorin) L.op.dev.gershgorin = est;
  }
  return 0;
}

int Hierarchy::build(pde_ctx* c, const Operator& fine, int kind, double p0, double p1) {
  release();
  const int dim = fine.g.dim;
  int ax[3], nax;
  internal_axes(dim, ax, &nax);
  int32_t n[3] = {0, 0, 0};
  double Lu[3] = {1, 1, 1};
  for (int q = 0; q < nax; ++q) {
    n[q] = fine.g.nc[ax[q]];
    Lu[q] = fine.g.h[ax[q]] * fine.g.nc[ax[q]];
  }
  const int ncomp = fine.tab.ncomp;
  // Slab runs: a level whose GLOBAL grid is small is replicated on every rank (and so are all coarser ones).  Its
  // right-hand side is assembled by one all-reduce of the restricted residual; the rest of the cycle below it runs
  // without any communication, instead of three latency-bound halo exchanges per level.
  static const long long rep_nodes = getenv("PDE_B200_REP_NODES") ? atoll(getenv("PDE_B200_REP_NODES")) : 400000;
  bool replicate = false;
  for (int level = 0;; ++level) {
    std::unique_ptr<MGLevel> L(new MGLevel());
    Grid g;
    if (c->world > 1 && level > 0 && !replicate) {
      long long gn = 1;
      for (int q = 0; q < nax; ++q) gn *= (n[q] + 1);
      replicate = gn <= rep_nodes;
    }
    if (replicate) {
      PDE_OK(make_grid(dim, n, Lu, 0, 1, &g));
      // only the FIRST replicated level is restricted into from a slab level and needs this rank's window; the
      // levels below may have fewer planes than ranks (a cubic 256^3 grid on 4 GPUs coarsens down to nz = 2)
      if (!lv.back()->replicated) {
        PDE_OK(make_grid(dim, n, Lu, c->rank, c->world, &L->gslab));
        L->gslab.comp_stride = g.comp_stride;   // a window into the replicated array: same pitch, rows and planes
      }
      L->replicated = true;
    } else {
      PDE_OK(make_grid(dim, n, Lu, c->rank, c->world, &g));
    }
    if (kind == PDE_OP_ELASTICITY) PDE_OK(L->op.setup_elasticity(c, g, fine.bc, p0, p1));
    else PDE_OK(L->op.setup_scalar(c, g, fine.bc, p0, p1));
    PDE_OK(L->xa.alloc(c, g, ncomp));
    PDE_OK(L->xb.alloc(c, g, ncomp));
    PDE_OK(L->r.alloc(c, g, ncomp));
    if (level > 0) PDE_OK(L->b.alloc(c, g, ncomp));
    lv.push_back(std::move(L));
    // can we coarsen further?
    bool can = true;
    if (const char* ml = getenv("PDE_B200_MAX_LEVELS")) can = can && (level + 1 < atoi(ml));
    int32_t nc2[3] = {0, 0, 0};
    // vector (elasticity) operators: re-discretised P1 operators on grids with a single cell across the body are
    // far too stiff in bending (locking), which spoils the coarse correction (33 -> ~20 PCG iterations on the
    // cantilever when the hierarchy stops at two cells across); scalar operators coarsen down to one cell
    static const int env_min = getenv("PDE_B200_MIN_COARSE_CELLS") ? atoi(getenv("PDE_B200_MIN_COARSE_CELLS")) : 0;
    const int min_cells = env_min > 0 ? env_min : (ncomp > 1 ? 2 : 1);
    for (int q = 0; q < nax; ++q) {
      if (n[q] % 2 != 0 || n[q] < 2) can = false;
      nc2[q] = n[q] / 2;
      if (nc2[q] < min_cells) can = false;
    }
    // slabs: the coarse partition must nest in the fine one (rank r owns coarse planes z0/2 ...)
    if (c->world > 1 && !replicate && n[nax - 1] % (2 * c->world) != 0) can = false;
    if (can) {
      Grid gc;
      PDE_OK(make_grid(dim, nc2, Lu, 0, 1, &gc));  // global view: every rank takes the same decision
      long long nodes = (long long)gc.nn[0] * gc.nn[1] * gc.nzl;
      if (nodes <= 200000) {
        long long nfree = count_free_and_index(gc, fine.bc, ncomp, nullptr, nullptr);
        if (nfree <= 0) can = false;
      }
    }
    if (!can) break;
    for (int q = 0; q < nax; ++q) n[q] = nc2[q];
  }
  // coarsest level: dense inverse if small enough
  MGLevel& Lc = *lv.back();
  long long nodes = (long long)Lc.op.g.nn[0] * Lc.op.g.nn[1] * Lc.op.g.nzg;
  if (lv.size() > 1 && nodes * ncomp <= 4 * PDE_DENSE_MAX) {
    Grid gg;
    PDE_OK(make_grid(dim, n, Lu, 0, 1, &gg));
    long long nfree = count_free_and_index(gg, Lc.op.bc, ncomp, nullptr, nullptr);
    if (nfree > 0 && nfree <= PDE_DENSE_MAX) PDE_OK(build_dense_coarse(c, Lc, dim, n, Lu));
  }
  if (ncomp > 1 && !getenv("PDE_B200_NO_LMAX_EST"))
    for (auto& L : lv) PDE_OK(estimate_lmax(c, *L, 12));
  return 0;
}

void Hierarchy::release() {
  if (gexec) cudaGraphExecDestroy(gexec);
  gexec = nullptr;
  gstate = 0;
  gnodes = 0;
  for (auto& L : lv) {
    L->op.release();
    L->b.release(); L->xa.release(); L->xb.release(); L->r.release();
    if (L->Ainv) cudaFree(L->Ainv);
    if (L->idx) cudaFree(L->idx);
    if (L->bglob) cudaFree(L->bglob);
  }
  lv.clear();
}

struct Cheby {
  double theta, delta, sigma, rho, lmax_;
  int kind = 1;  // 1: first-kind Chebyshev on [lmax/ratio, lmax]; 4: fourth-kind (Lottes), needs lmax only
  void init(double lmax, double ratio) {
    static const int env_kind = getenv("PDE_B200_CHEBY_KIND") ? atoi(getenv("PDE_B200_CHEBY_KIND")) : 1;
    kind = env_kind == 4 ? 4 : 1;
    lmax_ = lmax;
    const double lmin = lmax / ratio;
    theta = 0.5 * (lmax + lmin);
    delta = 0.5 * (lmax - lmin);
    sigma = theta / delta;
    rho = 1.0 / sigma;
  }
  // coefficients of sweep k (k = 0 restarts the recurrence): d = c1 d + c2 Dinv r
  void coef(int k, double* c1, double* c2) {
    if (kind == 4) {
      if (k == 0) { *c1 = 0.0; *c2 = 4.0 / (3.0 * lmax_); return; }
      *c1 = (2.0 * k - 1.0) / (2.0 * k + 3.0);
      *c2 = (8.0 * k + 4.0) / ((2.0 * k + 3.0) * lmax_);
      return;
    }
    if (k == 0) { rho = 1.0 / sigma; *c1 = 0.0; *c2 = 1.0 / theta; return; }
    const double rn = 1.0 / (2.0 * sigma - rho);
    *c1 = rn * rho;
    *c2 = 2.0 * rn / delta;
    rho = rn;
  }
};

// Chebyshev(Jacobi) smoothing.  dot_slot >= 0: the LAST sweep also leaves sum b.x_new in that scalar slot
// (*dot_done tells whether a sweep could do it).
static int smooth(pde_ctx* c, MGLevel& L, const double* b, double** cur, double** oth, int sweeps, bool zero_guess,
                  double ratio, int dot_slot = -1, bool* dot_done = nullptr, bool halos_valid = false) {
  Cheby ch;
  ch.init(L.op.dev.gershgorin, ratio);
  int k0 = 0;
  int prev_mode = 0;   // how sweep k rebuilds d_{k-1} = x_k - x_{k-1}
  double s0 = 0;
  if (dot_done) *dot_done = false;
  // vector operators with natural faces: k_elast3d + the two-layer face kernel (no fused dot product there)
  const bool e_first2 = !L.op.dev.uniform_diag && dot_slot < 0 && elast3d_first2_ok(L.op.g, L.op.bc, L.op.dev);
  if (zero_guess && sweeps >= 2 && (L.op.dev.uniform_diag || e_first2)) {
    // sweeps 0 and 1 in one pass over the data: x1 = s0 D^-1 b never touches memory
    StencilArgs a;
    double c1;
    ch.coef(0, &c1, &s0);
    a.cheby = 2;
    a.s0 = s0;
    ch.coef(1, &a.c1, &a.c2);
    a.x = b; a.y = *cur;
    if (dot_slot >= 0 && sweeps == 2) { a.reduce_slot_xy = dot_slot; if (dot_done) *dot_done = true; }
    if (c->world > 1) PDE_OK(comm_halo_exchange(c, L.op.g, L.op.dev.ncomp, const_cast<double*>(b)));
    PDE_OK(launch_stencil(c, L.op.g, L.op.bc, L.op.dev, a));
    L.paths |= PDE_MG_FIRST2;
    k0 = 2;
    prev_mode = 3;     // x_1 = s0 D^-1 b
  } else if (zero_guess) {
    double c1, c2;
    ch.coef(0, &c1, &c2);
    PDE_OK(launch_cheby_first(c, L.op.g, L.op.bc, L.op.dev, b, *cur, c2));
    k0 = 1;
    prev_mode = 2;     // x_0 = 0
  }
  // (the applicability test comes first: on slab levels too small for the fused kernels the two halo exchanges below
  // would be thrown away and repeated by the sweep loop)
  if (!zero_guess && sweeps == 2 && post2_applicable(L.op.g, L.op.dev) && (c->world == 1 || L.op.g.nzl >= PDE_NG)) {
    // both sweeps in one pass over the data (needs two halo planes of the iterate and one of the rhs)
    double c1a, c2a, c1b, c2b;
    ch.coef(0, &c1a, &c2a);
    ch.coef(1, &c1b, &c2b);
    bool handled = false;
    if (c->world > 1 && !halos_valid) {
      PDE_OK(comm_halo_exchange(c, L.op.g, 1, *cur, PDE_NG));
      PDE_OK(comm_halo_exchange(c, L.op.g, 1, const_cast<double*>(b), 1));
    }
    PDE_OK(launch_heat_post2(c, L.op.g, L.op.dev, *cur, b, *oth, c2a, c1b, c2b, dot_slot, &handled));
    if (handled) {
      L.paths |= PDE_MG_HEAT_POST2;
    } else {
      PDE_OK(launch_post2(c, L.op.g, L.op.bc, L.op.dev, *cur, b, *oth, c2a, c1b, c2b, dot_slot, &handled));
      if (handled) L.paths |= PDE_MG_POST2_R1;
    }
    if (handled) {
      std::swap(*cur, *oth);
      if (dot_slot >= 0 && dot_done) *dot_done = true;
      return 0;
    }
    ch.init(L.op.dev.gershgorin, ratio);  // not applicable: fall through to the separate sweeps
  }
  for (int k = k0; k < sweeps; ++k) {
    StencilArgs a;
    a.cheby = 1;
    a.x = *cur; a.y = *oth; a.b = b;
    ch.coef(k, &a.c1, &a.c2);
    a.prev_mode = k == 0 ? 0 : prev_mode;
    a.s0 = s0;
    a.xprev = a.prev_mode == 1 ? *oth : nullptr;   // the other buffer still holds x_{k-1}
    if (dot_slot >= 0 && k == sweeps - 1) { a.reduce_slot_xy = dot_slot; if (dot_done) *dot_done = true; }
    if (c->world > 1) PDE_OK(comm_halo_exchange(c, L.op.g, L.op.dev.ncomp, *cur));
    PDE_OK(launch_stencil(c, L.op.g, L.op.bc, L.op.dev, a));
    std::swap(*cur, *oth);
    prev_mode = 1;
  }
  return 0;
}

int Hierarchy::vcycle(pde_ctx* c, const Operator& fine, const double* b0, double** z_out, int dot_slot,
                      bool* dot_done) {
  if (dot_done) *dot_done = false;
  (void)fine;
  const int nl = (int)lv.size();
  std::vector<double*> cur(nl), oth(nl);
  for (int l = 0; l < nl; ++l) { cur[l] = lv[l]->xa.p; oth[l] = lv[l]->xb.p; }
  // slabs, uniform-diagonal scalar levels: the iterate is exchanged ONCE per level with two halo planes; residual
  // and prolongation are then computed on the ghost planes too, so neither the residual nor the corrected iterate
  // needs an exchange of its own (3 exchanges per level and cycle instead of 6)
  std::vector<char> lean(nl, 0);
  for (int l = 0; l + 1 < nl; ++l)
    lean[l] = c->world > 1 && !lv[l]->replicated && nu == 2 && lv[l]->op.dev.uniform_diag && lv[l]->op.dev.ncomp == 1 && lv[l]->op.g.dim == 3 &&
              lv[l]->op.g.nzl >= 8 && lv[l + 1]->op.g.nzl >= PDE_NG && sweep_applicable(lv[l]->op.g, 1) &&
              !getenv("PDE_B200_NO_POST2") && !getenv("PDE_B200_NO_LEAN_HALO");
  // down: pre-smoothing and residual of level l, restriction into level l+1
  auto down = [&](int l) -> int {
    MGLevel& L = *lv[l];
    const double* b = l == 0 ? b0 : L.b.p;
    PDE_OK(smooth(c, L, b, &cur[l], &oth[l], nu, true, ratio));   // exchanges one halo plane of b (fused first sweeps)
    if (c->world > 1) PDE_OK(comm_halo_exchange(c, L.op.g, L.op.dev.ncomp, cur[l], lean[l] ? PDE_NG : 1));
    return 0;
  };
  // residual of level l and its restriction into level l+1.  Uniform-diagonal scalar levels do both in one pass
  // (k_heat_post2<.., RR>: the fine residual never goes to HBM); otherwise residual kernel + restriction kernel.
  auto restrict_to = [&](int l) -> int {   // level l -> l+1
    MGLevel& L = *lv[l];
    MGLevel& Lc = *lv[l + 1];
    const double* b = l == 0 ? b0 : L.b.p;
    const bool window = Lc.replicated && !L.replicated;
    const Grid& gc = Lc.op.g;
    const int nc = L.op.dev.ncomp;
    // slab level -> replicated level: every rank restricts into its window of the global coarse array, the
    // windows are disjoint, one all-reduce (sum with zeros) completes the array everywhere
    if (window) PDE_OK(launch_zero(c, gc, nc, Lc.b.p));
    const Grid& gct = window ? Lc.gslab : gc;
    double* bct = window ? Lc.b.p + gc.plane * Lc.gslab.z0 : Lc.b.p;
    bool fused = false;
    if (c->world == 1 || lean[l]) PDE_OK(launch_heat_resid_restrict(c, L.op.g, gct, L.op.dev, cur[l], b, bct, &fused));
    if (fused) L.paths |= PDE_MG_RESID_RESTRICT;
    if (!fused) {
      StencilArgs a;
      a.x = cur[l]; a.b = b; a.y = L.r.p; a.bscale = 1.0; a.ascale = -1.0;
      a.ghost_out = lean[l];
      PDE_OK(launch_stencil(c, L.op.g, L.op.bc, L.op.dev, a));
      if (c->world > 1 && !lean[l]) PDE_OK(comm_halo_exchange(c, L.op.g, nc, L.r.p));
      PDE_OK(launch_restrict(c, L.op.g, gct, Lc.op.bc, nc, L.r.p, bct));
    }
    if (window) PDE_OK(comm_allreduce_buf(c, Lc.b.p, (size_t)(gc.comp_stride * (nc - 1) + gc.plane * gc.nzg)));
    return 0;
  };
  auto coarsest = [&]() -> int {
    MGLevel& L = *lv[nl - 1];
    const double* b = nl == 1 ? b0 : L.b.p;
    if (L.n_dense > 0 && (c->world == 1 || L.replicated)) {
      PDE_OK(launch_dense_solve(c, L.n_dense, L.Ainv, L.idx, b, cur[nl - 1]));
    } else if (L.n_dense > 0) {
      PDE_OK(launch_dense_gather(c, L.n_dense, L.idx, b, L.bglob));
      PDE_OK(comm_allreduce_buf(c, L.bglob, (size_t)L.n_dense));
      PDE_OK(launch_dense_solve_owned(c, L.n_dense, L.Ainv, L.idx, L.bglob, cur[nl - 1]));
    }
    else PDE_OK(smooth(c, L, b, &cur[nl - 1], &oth[nl - 1], nl == 1 ? nu : coarse_sweeps, true, nl == 1 ? ratio : 30.0,
                       nl == 1 ? dot_slot : -1, nl == 1 ? dot_done : nullptr));
    return 0;
  };
  auto prolong_into = [&](int l) -> int {   // level l+1 -> l
    MGLevel& L = *lv[l];
    if (c->world > 1) PDE_OK(comm_halo_exchange(c, lv[l + 1]->op.g, L.op.dev.ncomp, cur[l + 1], lean[l] ? PDE_NG : 1));
    PDE_OK(launch_prolong_add(c, L.op.g, lv[l + 1]->op.g, L.op.bc, L.op.dev.ncomp, cur[l + 1], cur[l], lean[l] ? PDE_NG : 0));
    return 0;
  };
  auto post = [&](int l) -> int {
    MGLevel& L = *lv[l];
    const double* b = l == 0 ? b0 : L.b.p;
    PDE_OK(smooth(c, L, b, &cur[l], &oth[l], nu, false, ratio, l == 0 ? dot_slot : -1, l == 0 ? dot_done : nullptr,
                  lean[l] != 0));
    return 0;
  };
  // The V-cycle on levels >= R (level R's right-hand side is ready): fixed kernels with fixed arguments and, when level R
  // is replicated (or on a single GPU), no communication at all - 40-60 launch-bound kernels that are captured into a
  // CUDA graph on the second cycle and replayed afterwards.
  auto sub = [&](int R) -> int {
    for (int l = R; l < nl - 1; ++l) { PDE_OK(down(l)); PDE_OK(restrict_to(l)); }
    PDE_OK(coarsest());
    for (int l = nl - 2; l >= R; --l) { PDE_OK(prolong_into(l)); PDE_OK(post(l)); }
    return 0;
  };
  // single GPU: R = 1 (the restriction out of level 0 and the prolongation back into it ride in the graph too);
  // slabs: R = the first replicated level (the levels above it exchange halos through flag-waiting kernels and NCCL,
  // which stay outside the graph)
  int R = 1;
  if (c->world > 1) {
    R = nl;
    for (int l = 1; l < nl; ++l)
      if (lv[l]->replicated) { R = l; break; }
  }
  const bool solo = c->world == 1;
  auto graph_part = [&]() -> int {
    if (solo) { PDE_OK(restrict_to(0)); PDE_OK(sub(1)); PDE_OK(prolong_into(0)); return 0; }
    // the prolongation out of level R rides along: it is the only reader of level R's result, whose buffer (the
    // ping-pong state after the smoother swaps) is only known while the sub-cycle is issued, not while it is replayed
    PDE_OK(sub(R));
    return prolong_into(R - 1);
  };
  auto run_graph_part = [&]() -> int {
    if (gstate == 2) {
      CUDA_OK(cudaGraphLaunch(gexec, c->stream));
      c->launches += gnodes;
    } else if (gstate == 1) {
      // second cycle: every static set-up (function attributes, tensor maps) happened in the first one
      const long long l0 = c->launches;
      CUDA_OK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
      const int rc = graph_part();
      cudaGraph_t graph = nullptr;
      const cudaError_t ec = cudaStreamEndCapture(c->stream, &graph);
      if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (ec != cudaSuccess || !graph) { cudaGetLastError(); gstate = -1; PDE_OK(graph_part()); }
      else {
        gnodes = c->launches - l0;
        const cudaError_t ei = cudaGraphInstantiate(&gexec, graph, 0);
        cudaGraphDestroy(graph);
        if (ei != cudaSuccess) { cudaGetLastError(); gexec = nullptr; gstate = -1; c->launches = l0; PDE_OK(graph_part()); }
        else {
          gstate = 2;
          CUDA_OK(cudaGraphLaunch(gexec, c->stream));   // the capture did not execute anything
        }
      }
    } else {
      PDE_OK(graph_part());
      if (gstate == 0) gstate = 1;
    }
    return 0;
  };
  if (nl == 1) {
    PDE_OK(coarsest());
    *z_out = cur[0];
    return 0;
  }
  static const int graph_env = getenv("PDE_B200_MG_GRAPH") ? atoi(getenv("PDE_B200_MG_GRAPH")) : 1;
  if (gstate == 0 && !(graph_env && (solo ? nl >= 3 : nl - R >= 2))) gstate = -1;
  PDE_OK(down(0));
  if (solo) {
    PDE_OK(run_graph_part());
  } else {
    PDE_OK(restrict_to(0));
    for (int l = 1; l < R && l < nl - 1; ++l) { PDE_OK(down(l)); PDE_OK(restrict_to(l)); }
    if (R < nl) {
      PDE_OK(run_graph_part());
      for (int l = R - 1; l >= 1; --l) { PDE_OK(post(l)); PDE_OK(prolong_into(l - 1)); }
    } else {          // no replicated level: the coarsest level is a slab level
      PDE_OK(coarsest());
      for (int l = nl - 2; l >= 1; --l) { PDE_OK(prolong_into(l)); PDE_OK(post(l)); }
      PDE_OK(prolong_into(0));
    }
  }
  PDE_OK(post(0));
  *z_out = cur[0];
  return 0;
}

int choose_precond(const pde_solver_opts& o, pde_ctx* c, long long ndofs, const Hierarchy& h) {
  if (o.precond == PDE_PRECOND_JACOBI) return PDE_PRECOND_JACOBI;
  if (h.levels() < 2) return PDE_PRECOND_JACOBI;
  if (o.precond == PDE_PRECOND_GMG) return PDE_PRECOND_GMG;
  (void)c;
  return ndofs >= 20000 ? PDE_PRECOND_GMG : PDE_PRECOND_JACOBI;
}

// ---- PCG -----------------------------------------------------------------------------------------
int PcgWork::alloc(pde_ctx* c, const Grid& g, int ncomp) {
  PDE_OK(p.alloc(c, g, ncomp));
  PDE_OK(q.alloc(c, g, ncomp));
  return 0;
}
void PcgWork::release() { p.release(); q.release(); }

int pcg_solve(pde_ctx* c, const Operator& A, Hierarchy* mg, PcgWork& w, double* x, double* r, double bnorm2,
              const pde_solver_opts& o, pde_stats* st) {
  const Grid& g = A.g;
  const int nc = A.dev.ncomp;
  const bool gmg = mg != nullptr;
  const double tol2 = o.rtol * o.rtol * bnorm2;
  st->solves += 1;
  st->levels = gmg ? mg->levels() : 1;
  if (!(bnorm2 > 0.0)) {  // zero right-hand side: the initial guess (Dirichlet lift) is the solution
    st->final_relres = 0.0;
    return 0;
  }
  double* z = nullptr;
  double rr;
  if (!gmg) {
    CUDA_OK(cudaMemsetAsync(c->scal + S_XY, 0, 2 * sizeof(double), c->stream));
    PDE_OK(launch_cg_update(c, g, A.dev, x, r, w.p.p, w.q.p, S_RHO0, S_XY, S_RHO0, S_RHO0 + 1, 1));
    if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_RHO0, 2));
    PDE_OK(launch_cg_pupdate(c, g, A.dev, w.p.p, r, S_RHO0, S_RHO0, 1, 1));
  } else {
    bool fused = false;
    PDE_OK(mg->vcycle(c, A, r, &z, S_RHO0, &fused));
    if (!fused) PDE_OK(launch_dot(c, g, nc, r, z, S_RHO0));
    PDE_OK(launch_dot(c, g, nc, r, r, S_RHO0 + 1));
    if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_RHO0, 2));
    PDE_OK(launch_cg_pupdate(c, g, A.dev, w.p.p, z, S_RHO0, S_RHO0, 1, 0));
  }
  PDE_OK(read_scal(c, S_RHO0 + 1, 1, &rr));
  const bool trace = getenv("PDE_B200_TRACE") != nullptr;
  if (trace) {
    double v[2];
    PDE_OK(read_scal(c, S_RHO0, 2, v));
    fprintf(stderr, "[pcg] n=%lld gmg=%d levels=%d bnorm2=%.6e rho0=%.6e rr0=%.6e\n", (long long)g.total, (int)gmg,
            gmg ? mg->levels() : 1, bnorm2, v[0], v[1]);
  }
  int it = 0;
  bool conv = rr <= tol2;
  const int check = gmg ? 1 : (o.check_every > 0 ? o.check_every : 10);
  while (!conv && it < o.max_iters) {
    const int sr = 2 * (it & 1), sn = 2 * (1 - (it & 1));
    StencilArgs a;
    a.x = w.p.p; a.y = w.q.p; a.reduce_slot_xy = S_XY;
    a.skip_yy = 1;   // only p.Ap is needed
    if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, w.p.p));
    PDE_OK(launch_stencil(c, g, A.bc, A.dev, a));
    if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_XY, 1));
    // GMG path: x += alpha p is deferred to the p update below (p is read there anyway)
    PDE_OK(launch_cg_update(c, g, A.dev, gmg ? nullptr : x, r, w.p.p, w.q.p, sr, S_XY, sn, sn + 1, !gmg));
    // slots (sn, sn+1) = (r.z, r.r): Jacobi fills both in the update kernel; with multigrid r.z only exists after
    // the V-cycle, so the two partial sums travel in ONE all-reduce there (r.r is only needed by the poll below)
    if (c->world > 1 && !gmg) PDE_OK(comm_allreduce_scal(c, sn, 2));
    if (gmg) {
      bool fused = false;
      PDE_OK(mg->vcycle(c, A, r, &z, sn, &fused));
      if (!fused) PDE_OK(launch_dot(c, g, nc, r, z, sn));
      if (c->world > 1) PDE_OK(comm_allreduce_scal(c, sn, 2));
    }
    PDE_OK(launch_cg_pupdate(c, g, A.dev, w.p.p, gmg ? z : r, sr, sn, 0, !gmg, gmg ? x : nullptr, S_XY));
    ++it;
    if (trace && (it <= 30 || it % 50 == 0)) {
      double v[2], pap;
      PDE_OK(read_scal(c, sn, 2, v));
      PDE_OK(read_scal(c, S_XY, 1, &pap));
      fprintf(stderr, "[pcg] it=%d pAp=%.6e rho=%.6e rr=%.6e\n", it, pap, v[0], v[1]);
    }
    if (it % check == 0 || it >= o.max_iters) {
      PDE_OK(read_scal(c, sn + 1, 1, &rr));
      if (!(rr == rr)) PDE_FAIL("PCG broke down (NaN residual)");
      conv = rr <= tol2;
    }
  }
  st->iters_total += it;
  st->final_relres = std::sqrt(rr / bnorm2);
  if (!conv) st->converged = 0;
  return 0;
}
