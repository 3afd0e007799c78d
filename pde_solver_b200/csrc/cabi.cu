// extern "C" entry points of libpde_b200.so (see include/pde_b200.h for the reference interface each
// one replaces).  No torch types, no callbacks, no stdout.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#include "solver.cuh"

int comm_destroy(pde_ctx* c);

// ---- context ----------------------------------------------------------------------------------
extern "C" int pde_ctx_create(int device, pde_ctx** out) {
  if (!out) PDE_FAIL("null out pointer");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    PDE_FAIL(std::string("no CUDA device available (this library has no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= ndev) PDE_FAIL("device index out of range");
  CUDA_OK(cudaSetDevice(device));
  pde_ctx* c = new (std::nothrow) pde_ctx();
  if (!c) PDE_FAIL("out of host memory");
  c->device = device;
  cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
  CUDA_OK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CUDA_OK(cudaEventCreate(&c->ev0));
  CUDA_OK(cudaEventCreate(&c->ev1));
  CUDA_OK(cudaEventCreateWithFlags(&c->ev_poll, cudaEventDisableTiming));
  CUDA_OK(cudaMalloc(&c->red.partials, sizeof(double) * RED_MAX_BLOCKS * RED_MAX_VALS));
  CUDA_OK(cudaMalloc(&c->red.counter, sizeof(unsigned)));
  CUDA_OK(cudaMalloc(&c->face_partials, sizeof(double) * RED_MAX_BLOCKS * RED_MAX_VALS));
  CUDA_OK(cudaMemsetAsync(c->red.counter, 0, sizeof(unsigned), c->stream));
  CUDA_OK(cudaMalloc(&c->scal, sizeof(double) * S_NSLOTS));
  CUDA_OK(cudaMemsetAsync(c->scal, 0, sizeof(double) * S_NSLOTS, c->stream));
  CUDA_OK(cudaStreamSynchronize(c->stream));
  CUDA_OK(cudaHostAlloc(&c->h_scal, sizeof(double) * S_NSLOTS, cudaHostAllocMapped));
  *out = c;
  return 0;
}

extern "C" int pde_ctx_destroy(pde_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  comm_destroy(c);
  cudaFree(c->red.partials);
  cudaFree(c->red.counter);
  cudaFree(c->face_partials);
  if (c->scratch) cudaFree(c->scratch);
  cudaFree(c->scal);
  cudaFreeHost(c->h_scal);
  cudaEventDestroy(c->ev0);
  cudaEventDestroy(c->ev1);
  cudaEventDestroy(c->ev_poll);
  cudaStreamDestroy(c->stream);
  delete c;
  return 0;
}

extern "C" int64_t pde_ctx_launch_count(pde_ctx* c) { return c ? c->launches : 0; }
extern "C" int pde_ctx_sync(pde_ctx* c) {
  CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}
extern "C" int pde_timer_start(pde_ctx* c) {
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  return 0;
}
extern "C" int pde_timer_stop(pde_ctx* c, double* ms) {
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float f = 0;
  CUDA_OK(cudaEventElapsedTime(&f, c->ev0, c->ev1));
  if (ms) *ms = f;
  return 0;
}

extern "C" int pde_host_alloc(uint64_t bytes, void** out) {
  if (!out) PDE_FAIL("null out pointer");
  CUDA_OK(cudaHostAlloc(out, bytes ? bytes : 8, cudaHostAllocDefault));
  return 0;
}
extern "C" int pde_host_free(void* p) {
  if (p) CUDA_OK(cudaFreeHost(p));
  return 0;
}

struct DevMem {
  void* p = nullptr;
  ~DevMem() { if (p) cudaFree(p); }
  int alloc(size_t bytes) {
    CUDA_OK(cudaMalloc(&p, bytes ? bytes : 8));
    return 0;
  }
};

extern "C" int pde_halo_bench(pde_ctx* c, int dim, const int32_t n[3], int ncomp, int reps, double* ms_per_exchange,
                              int64_t* bytes_sent) {
  if (!c) PDE_FAIL("null context");
  if (ncomp < 1 || ncomp > 3) PDE_FAIL("ncomp must be 1..3");
  CUDA_OK(cudaSetDevice(c->device));
  const double L1[3] = {1, 1, 1};
  Grid g;
  PDE_OK(make_grid(dim, n, L1, c->rank, c->world, &g));
  Field f;
  struct Rel { Field* f; ~Rel() { f->release(); } } rel{&f};
  PDE_OK(f.alloc(c, g, ncomp));
  for (int i = 0; i < 3; ++i) PDE_OK(comm_halo_exchange(c, g, ncomp, f.p));
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  for (int i = 0; i < reps; ++i) PDE_OK(comm_halo_exchange(c, g, ncomp, f.p));
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  if (ms_per_exchange) *ms_per_exchange = ms / (reps > 0 ? reps : 1);
  const int nbr = (c->rank > 0 ? 1 : 0) + (c->rank < c->world - 1 ? 1 : 0);
  if (bytes_sent) *bytes_sent = (int64_t)nbr * ncomp * g.plane * (int64_t)sizeof(double);
  return 0;
}

// Halo exchange self-check: a field whose values depend on the GLOBAL node index is exchanged `reps` times with
// `depth` planes (scaled by 2 and with the ghost planes wiped between repetitions, so stale or misplaced planes
// show); *mismatches = number of ghost entries that differ bitwise from the owner's value.
extern "C" int pde_halo_check(pde_ctx* c, int dim, const int32_t n[3], int ncomp, int depth, int reps,
                              int64_t* mismatches) {
  if (!c || !mismatches) PDE_FAIL("null argument");
  if (ncomp < 1 || ncomp > 3) PDE_FAIL("ncomp must be 1..3");
  if (depth < 1 || depth > PDE_NG) PDE_FAIL("depth out of range");
  CUDA_OK(cudaSetDevice(c->device));
  const double L1[3] = {1, 1, 1};
  Grid g;
  PDE_OK(make_grid(dim, n, L1, c->rank, c->world, &g));
  Field f;
  struct Rel { Field* f; ~Rel() { f->release(); } } rel{&f};
  PDE_OK(f.alloc(c, g, ncomp));
  DevMem bad;
  PDE_OK(bad.alloc(sizeof(unsigned long long)));
  CUDA_OK(cudaMemsetAsync(bad.p, 0, sizeof(unsigned long long), c->stream));
  BcDev nobc;
  std::memset(&nobc, 0, sizeof(nobc));
  PDE_OK(launch_fill_pattern(c, g, nobc, ncomp, f.p));
  double scale = 1.0;
  for (int r = 0; r < reps; ++r) {
    for (int i = 0; i < ncomp; ++i) {   // wipe the ghost planes
      double* b = f.p + (size_t)i * g.comp_stride;
      CUDA_OK(cudaMemsetAsync(b - (size_t)PDE_NG * g.plane, 0, sizeof(double) * PDE_NG * g.plane, c->stream));
      CUDA_OK(cudaMemsetAsync(b + (size_t)g.nzl * g.plane, 0, sizeof(double) * PDE_NG * g.plane, c->stream));
    }
    PDE_OK(comm_halo_exchange(c, g, ncomp, f.p, depth));
    PDE_OK(launch_halo_verify(c, g, ncomp, depth, f.p, scale, (unsigned long long*)bad.p));
    PDE_OK(launch_axpy(c, g, ncomp, f.p, f.p, 1.0));   // f <- 2 f (owned planes; exact)
    scale *= 2.0;
  }
  unsigned long long nb = 0;
  PDE_OK(d2h(c, &nb, bad.p, sizeof(nb)));
  if (c->world > 1) PDE_OK(comm_check_error(c));
  *mismatches = (int64_t)nb;
  return 0;
}

// ---- meshes -------------------------------------------------------------------------------------
extern "C" int pde_mesh_coords(pde_ctx* c, int dim, const int32_t n[3], const double L[3], double* coords) {
  if (!c) PDE_FAIL("null context");
  CUDA_OK(cudaSetDevice(c->device));
  int64_t nv, nc;
  PDE_OK(pde_mesh_counts(dim, n, &nv, &nc));
  DevMem d;
  PDE_OK(d.alloc(sizeof(double) * nv * dim));
  PDE_OK(launch_mesh_coords(c, dim, n, L, (double*)d.p));
  return d2h(c, coords, d.p, sizeof(double) * nv * dim);
}

extern "C" int pde_mesh_coords_box(pde_ctx* c, int dim, const int32_t n[3], const double lo[3], const double hi[3],
                                   double* coords) {
  if (!c) PDE_FAIL("null context");
  CUDA_OK(cudaSetDevice(c->device));
  int64_t nv, nc;
  PDE_OK(pde_mesh_counts(dim, n, &nv, &nc));
  DevMem d;
  PDE_OK(d.alloc(sizeof(double) * nv * dim));
  PDE_OK(launch_mesh_coords_box(c, dim, n, lo, hi, (double*)d.p));
  return d2h(c, coords, d.p, sizeof(double) * nv * dim);
}

extern "C" int pde_dofmap_cells(pde_ctx* c, int dim, const int32_t n[3], int ncomp, int layout, int32_t* out) {
  if (!c) PDE_FAIL("null context");
  if (ncomp < 1 || ncomp > 3) PDE_FAIL("ncomp must be 1..3");
  CUDA_OK(cudaSetDevice(c->device));
  int64_t nv, nc;
  PDE_OK(pde_mesh_counts(dim, n, &nv, &nc));
  if (nv * ncomp > 2147483647LL) PDE_FAIL("dof indices exceed int32; export connectivity at smaller sizes only");
  DevMem d;
  size_t bytes = sizeof(int32_t) * nc * (dim + 1) * ncomp;
  PDE_OK(d.alloc(bytes));
  PDE_OK(launch_mesh_cells(c, dim, n, /*sorted=*/1, ncomp, layout, (int32_t*)d.p));
  return d2h(c, out, d.p, bytes);
}

extern "C" int pde_mesh_cells(pde_ctx* c, int dim, const int32_t n[3], int sorted, int32_t* cells) {
  if (!c) PDE_FAIL("null context");
  CUDA_OK(cudaSetDevice(c->device));
  int64_t nv, nc;
  PDE_OK(pde_mesh_counts(dim, n, &nv, &nc));
  if (nv > 2147483647LL) PDE_FAIL("vertex indices exceed int32");
  DevMem d;
  size_t bytes = sizeof(int32_t) * nc * (dim + 1);
  PDE_OK(d.alloc(bytes));
  PDE_OK(launch_mesh_cells(c, dim, n, sorted, 1, 0, (int32_t*)d.p));
  return d2h(c, cells, d.p, bytes);
}

static int make_bc(int dim, const int32_t n[3], const pde_bc* bc, BcDev* out) {
  user_bc_to_dev(dim, bc, out);
  if (out->side_excl && n[0] < 3) {  // every side facet touches an x-end: the topological set is empty
    for (int f = 2; f < 6; ++f) out->on[f] = 0;
  }
  return 0;
}

extern "C" int pde_boundary_mask(pde_ctx* c, int dim, const int32_t n[3], const pde_bc* bc, uint8_t* mask,
                                 double* vals) {
  if (!c) PDE_FAIL("null context");
  CUDA_OK(cudaSetDevice(c->device));
  const double L1[3] = {1, 1, 1};
  Grid g;
  PDE_OK(make_grid(dim, n, L1, 0, 1, &g));
  BcDev b;
  PDE_OK(make_bc(dim, n, bc, &b));
  int64_t nv, nc;
  PDE_OK(pde_mesh_counts(dim, n, &nv, &nc));
  DevMem dm, dv;
  PDE_OK(dm.alloc(nv));
  PDE_OK(dv.alloc(sizeof(double) * nv));
  PDE_OK(launch_bc_mask(c, g, b, (uint8_t*)dm.p, vals ? (double*)dv.p : nullptr));
  PDE_OK(d2h(c, mask, dm.p, nv));
  if (vals) PDE_OK(d2h(c, vals, dv.p, sizeof(double) * nv));
  return 0;
}

// ---- heat ---------------------------------------------------------------------------------------
struct pde_heat_state {
  pde_ctx* c = nullptr;
  pde_heat_params p{};
  pde_solver_opts o{};
  Grid g{};
  BcDev bc{};
  Operator A, K, M;
  Hierarchy mg;
  bool use_mg = false;
  PcgWork w;
  Field u, r;
  Field un;               // u_n of a verified solve (true-residual check), allocated on first use
  DevMem dense;
  long long nloc = 0;
  double setup_ms = 0;
  // copy pipeline (pde_heat_advance_batch, snapshots of pde_heat_solve): two staging buffers per direction and one
  // stream per direction, so that PCIe traffic in both directions overlaps the solve on the compute stream
  struct Pipe {
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaEvent_t in_ready[2] = {}, in_free[2] = {}, out_ready[2] = {}, out_free[2] = {};
    double* in[2] = {nullptr, nullptr};
    double* out[2] = {nullptr, nullptr};
    long long nout = 0;      // snapshots handed to the d2h stream so far
    bool ready = false;
  } pipe;
};

static void pipe_release(pde_heat_state* s) {
  pde_heat_state::Pipe& q = s->pipe;
  if (q.h2d) { cudaStreamSynchronize(q.h2d); cudaStreamDestroy(q.h2d); }
  if (q.d2h) { cudaStreamSynchronize(q.d2h); cudaStreamDestroy(q.d2h); }
  for (int i = 0; i < 2; ++i) {
    if (q.in_ready[i]) cudaEventDestroy(q.in_ready[i]);
    if (q.in_free[i]) cudaEventDestroy(q.in_free[i]);
    if (q.out_ready[i]) cudaEventDestroy(q.out_ready[i]);
    if (q.out_free[i]) cudaEventDestroy(q.out_free[i]);
    if (q.in[i]) cudaFree(q.in[i]);
    if (q.out[i]) cudaFree(q.out[i]);
  }
  q = pde_heat_state::Pipe();
}

static int pipe_init(pde_heat_state* s, bool want_in) {
  pde_heat_state::Pipe& q = s->pipe;
  if (!q.ready) {
    CUDA_OK(cudaStreamCreateWithFlags(&q.h2d, cudaStreamNonBlocking));
    CUDA_OK(cudaStreamCreateWithFlags(&q.d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CUDA_OK(cudaEventCreateWithFlags(&q.in_ready[i], cudaEventDisableTiming));
      CUDA_OK(cudaEventCreateWithFlags(&q.in_free[i], cudaEventDisableTiming));
      CUDA_OK(cudaEventCreateWithFlags(&q.out_ready[i], cudaEventDisableTiming));
      CUDA_OK(cudaEventCreateWithFlags(&q.out_free[i], cudaEventDisableTiming));
      CUDA_OK(cudaMalloc((void**)&q.out[i], sizeof(double) * (s->nloc ? s->nloc : 1)));
    }
    q.ready = true;
  }
  if (want_in && !q.in[0])
    for (int i = 0; i < 2; ++i) CUDA_OK(cudaMalloc((void**)&q.in[i], sizeof(double) * (s->nloc ? s->nloc : 1)));
  return 0;
}

// pack the current state into a staging buffer on the compute stream and hand it to the d2h stream; returns
// without waiting for the copy (pipe_drain waits)
static int pipe_push_snapshot(pde_heat_state* s, double* dst_host) {
  pde_ctx* c = s->c;
  pde_heat_state::Pipe& q = s->pipe;
  const int b = (int)(q.nout & 1);
  if (q.nout >= 2) CUDA_OK(cudaStreamWaitEvent(c->stream, q.out_free[b], 0));
  PDE_OK(launch_pack(c, s->g, 1, s->u.p, q.out[b], 0));
  CUDA_OK(cudaEventRecord(q.out_ready[b], c->stream));
  CUDA_OK(cudaStreamWaitEvent(q.d2h, q.out_ready[b], 0));
  CUDA_OK(cudaMemcpyAsync(dst_host, q.out[b], sizeof(double) * s->nloc, cudaMemcpyDeviceToHost, q.d2h));
  CUDA_OK(cudaEventRecord(q.out_free[b], q.d2h));
  q.nout += 1;
  return 0;
}

static int pipe_drain(pde_heat_state* s) {
  if (s->pipe.h2d) CUDA_OK(cudaStreamSynchronize(s->pipe.h2d));
  if (s->pipe.d2h) CUDA_OK(cudaStreamSynchronize(s->pipe.d2h));
  return 0;
}

extern "C" int pde_heat_close(pde_heat_state* s) {
  if (!s) return 0;
  cudaSetDevice(s->c->device);
  cudaStreamSynchronize(s->c->stream);
  pipe_release(s);
  s->A.release(); s->K.release(); s->M.release();
  s->mg.release();
  s->w.release();
  s->u.release(); s->r.release(); s->un.release();
  delete s;
  return 0;
}

extern "C" int pde_heat_open(pde_ctx* c, const pde_heat_params* p, const pde_solver_opts* o, pde_heat_state** out) {
  if (!c || !p || !out) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(c->device));
  if (!p->steady && !(p->dt > 0)) PDE_FAIL("dt must be > 0");
  if (!(p->diffusivity > 0)) PDE_FAIL("diffusivity must be > 0");
  if (p->num_steps < 0) PDE_FAIL("num_steps must be >= 0");
  pde_heat_state* s = new (std::nothrow) pde_heat_state();
  if (!s) PDE_FAIL("out of host memory");
  s->c = c;
  s->p = *p;
  if (o) s->o = *o; else pde_solver_opts_default(&s->o);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  cudaEventRecord(e0, c->stream);
  int rc = 0;
  do {
    if ((rc = make_grid(p->dim, p->n, p->L, c->rank, c->world, &s->g))) break;
    if ((rc = make_bc(p->dim, p->n, &p->bc, &s->bc))) break;
    const double kappa = p->diffusivity;
    const double alpha = p->steady ? 0.0 : 1.0, beta = p->steady ? kappa : p->dt * kappa;
    if ((rc = s->A.setup_scalar(c, s->g, s->bc, alpha, beta))) break;
    if ((rc = s->K.setup_scalar(c, s->g, s->bc, 0.0, 1.0))) break;
    if ((rc = s->M.setup_scalar(c, s->g, s->bc, 1.0, 0.0))) break;
    if ((rc = s->u.alloc(c, s->g, 1))) break;
    if ((rc = s->r.alloc(c, s->g, 1))) break;
    if ((rc = s->w.alloc(c, s->g, 1))) break;
    s->nloc = (long long)s->g.nn[0] * s->g.nn[1] * s->g.nzl;
    if ((rc = s->dense.alloc(sizeof(double) * s->nloc))) break;
    long long ndofs = (long long)s->g.nn[0] * s->g.nn[1] * s->g.nzg;
    if (s->o.precond != PDE_PRECOND_JACOBI) {
      if ((rc = s->mg.build(c, s->A, PDE_OP_HEAT, alpha, beta))) break;
      s->mg.nu = s->o.cheby_degree > 0 ? s->o.cheby_degree : 2;
      s->mg.ratio = s->o.cheby_ratio > 1 ? s->o.cheby_ratio : 8.0;
    }
    s->use_mg = choose_precond(s->o, c, ndofs, s->mg) == PDE_PRECOND_GMG;
    if (!s->use_mg) s->mg.release();
    // initial condition (reference :276-297, 408-426, 672-691): fill, then bc.apply(u_n.vector())
    double v0 = p->initial_type == PDE_IC_ZERO ? 0.0 : p->T_initial;
    if (p->steady) v0 = 0.0;
    if (!p->steady && (p->initial_type == PDE_IC_COSINE || p->initial_type == PDE_IC_SINE)) {
      if ((rc = project_trig_ic(c, s->g, s->bc, p->dim, p->n, p->L, nullptr, p->initial_amplitude,
                                p->initial_wavenumber, p->initial_type == PDE_IC_SINE, s->o, s->u.p, s->r.p))) break;
    } else {
      if ((rc = launch_fill_ic(c, s->g, s->bc, s->u.p, v0, 1))) break;
    }
  } while (0);
  cudaEventRecord(e1, c->stream);
  cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  s->setup_ms = ms;
  if (rc) { pde_heat_close(s); return rc; }
  *out = s;
  return 0;
}

extern "C" int64_t pde_heat_local_nverts(pde_heat_state* s) { return s ? s->nloc : 0; }

extern "C" int pde_heat_set_state(pde_heat_state* s, const double* u_host) {
  if (!s || !u_host) PDE_FAIL("null argument");
  pde_ctx* c = s->c;
  CUDA_OK(cudaSetDevice(c->device));
  CUDA_OK(cudaMemcpyAsync(s->dense.p, u_host, sizeof(double) * s->nloc, cudaMemcpyHostToDevice, c->stream));
  PDE_OK(launch_unpack(c, s->g, 1, (const double*)s->dense.p, s->u.p, 0));
  PDE_OK(launch_apply_bc_values(c, s->g, s->bc, s->u.p));
  return 0;
}

extern "C" int pde_heat_get_state(pde_heat_state* s, double* u_host) {
  if (!s || !u_host) PDE_FAIL("null argument");
  pde_ctx* c = s->c;
  CUDA_OK(cudaSetDevice(c->device));
  PDE_OK(launch_pack(c, s->g, 1, s->u.p, (double*)s->dense.p, 0));
  return d2h(c, u_host, s->dense.p, sizeof(double) * s->nloc);
}

// verify: also recompute the true residual ||b - A u_{n+1}|| / ||b|| of this solve (st->true_relres) instead of
// trusting the PCG recurrence (SURVEY hard part 3).  Costs one copy of u_n and two operator applications.
static int heat_one_solve(pde_heat_state* s, pde_stats* st, bool verify = false) {
  pde_ctx* c = s->c;
  const pde_heat_params& p = s->p;
  const double f = p.source_value, kappa = p.diffusivity;
  if (verify && !p.steady) {
    if (!s->un.p) PDE_OK(s->un.alloc(c, s->g, 1));
    PDE_OK(launch_copy(c, s->g, 1, s->un.p, s->u.p));
  }
  // r0.r0 (for pcg_solve's first convergence test) comes from the pass that writes r0, into S_RHO1; ||b||^2 goes to
  // S_RR, so one all-reduce and one poll carry both.  Slots S_RHO0 .. S_RR are free until PCG writes them.
  StencilArgs a;
  a.x = s->u.p; a.y = s->r.p; a.bconst[0] = f; a.reduce_slot_xy = S_RHO0;
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, s->g, 1, s->u.p));
  double rr0, bn2;
  if (p.steady) {
    // r0 = f m - kappa K u0 (u0 = Dirichlet lift): this IS the reduced right-hand side, ||b||^2 = r0.r0
    a.bscale = 1.0; a.ascale = -1.0;
    PDE_OK(launch_stencil(c, s->g, s->bc, s->A.dev, a));
    if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_RHO1, 1));
    PDE_OK(read_scal(c, S_RHO1, 1, &rr0));
    bn2 = rr0;
  } else {
    // warm start x0 = u_n  =>  r0 = b - A u_n = dt (f m - kappa K u_n)   (b = M u_n + dt f m)
    a.bscale = p.dt; a.ascale = -p.dt * kappa;
    PDE_OK(launch_stencil(c, s->g, s->bc, s->K.dev, a));
    StencilArgs nb;   // b: u.b into S_PAP, ||b||^2 into S_RR
    nb.x = s->u.p; nb.y = nullptr; nb.bconst[0] = f; nb.bscale = p.dt; nb.ascale = 1.0; nb.reduce_slot_xy = S_PAP;
    PDE_OK(launch_stencil(c, s->g, s->bc, s->M.dev, nb));
    static_assert(S_RR == S_RHO1 + 2, "r0.r0 and ||b||^2 are read in one call");
    if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_RHO1, 3));
    double v[3];
    PDE_OK(read_scal(c, S_RHO1, 3, v));
    rr0 = v[0];
    bn2 = v[2];
  }
  PDE_OK(pcg_solve(c, s->A, s->use_mg ? &s->mg : nullptr, s->w, s->u.p, s->r.p, bn2, s->o, st, &rr0));
  if (verify) {
    StencilArgs t;
    t.y = s->r.p; t.reduce_slot_xy = S_XY;
    if (c->world > 1) PDE_OK(comm_halo_exchange(c, s->g, 1, s->u.p));
    if (p.steady) {   // residual of the reduced system: f m - kappa K u on the free rows
      t.x = s->u.p; t.bconst[0] = f; t.bscale = 1.0; t.ascale = -1.0;
      PDE_OK(launch_stencil(c, s->g, s->bc, s->A.dev, t));
    } else {          // b = M u_n + dt f m, then b - A u_{n+1}
      if (c->world > 1) PDE_OK(comm_halo_exchange(c, s->g, 1, s->un.p));
      StencilArgs tb;
      tb.x = s->un.p; tb.y = s->r.p; tb.bconst[0] = f; tb.bscale = p.dt; tb.ascale = 1.0;
      PDE_OK(launch_stencil(c, s->g, s->bc, s->M.dev, tb));
      t.x = s->u.p; t.b = s->r.p; t.bscale = 1.0; t.ascale = -1.0;
      PDE_OK(launch_stencil(c, s->g, s->bc, s->A.dev, t));
    }
    if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_XY, 2));
    double rr;
    PDE_OK(read_scal(c, S_YY, 1, &rr));
    st->true_relres = bn2 > 0 ? std::sqrt(rr / bn2) : 0.0;
  }
  return 0;
}

static void stats_init(pde_stats* st, long long ndofs) {
  std::memset(st, 0, sizeof(*st));
  st->ndofs = ndofs;
  st->converged = 1;
  st->true_relres = NAN;
}

extern "C" int pde_heat_step(pde_heat_state* s, int nsteps, pde_stats* st_out) {
  if (!s) PDE_FAIL("null state");
  pde_ctx* c = s->c;
  CUDA_OK(cudaSetDevice(c->device));
  pde_stats st;
  stats_init(&st, (long long)s->g.nn[0] * s->g.nn[1] * s->g.nzg);
  const long long l0 = c->launches;
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  for (int k = 0; k < nsteps; ++k) {
    PDE_OK(heat_one_solve(s, &st, k == nsteps - 1 && s->o.verify_residual >= 0));
  }
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  st.solve_ms = ms;
  st.setup_ms = s->setup_ms;
  st.launches = c->launches - l0;
  if (st_out) *st_out = st;
  return 0;
}

// A batch of independent one-step advances u_in[k] -> u_out[k] with HOST buffers (pinned for full overlap): the
// upload of request k+1 and the download of result k-1 run on their own streams while request k is solved.
extern "C" int pde_heat_advance_batch(pde_heat_state* s, int nreq, const double* const* u_in_host,
                                      double* const* u_out_host, pde_stats* st_out) {
  if (!s || !u_in_host || !u_out_host) PDE_FAIL("null argument");
  if (nreq < 0) PDE_FAIL("nreq must be >= 0");
  pde_ctx* c = s->c;
  CUDA_OK(cudaSetDevice(c->device));
  PDE_OK(pipe_init(s, true));
  pde_heat_state::Pipe& q = s->pipe;
  pde_stats st;
  stats_init(&st, (long long)s->g.nn[0] * s->g.nn[1] * s->g.nzg);
  const long long l0 = c->launches;
  const size_t bytes = sizeof(double) * s->nloc;
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  q.nout = 0;
  if (nreq > 0) {
    if (!u_in_host[0]) PDE_FAIL("null input buffer");
    CUDA_OK(cudaMemcpyAsync(q.in[0], u_in_host[0], bytes, cudaMemcpyHostToDevice, q.h2d));
    CUDA_OK(cudaEventRecord(q.in_ready[0], q.h2d));
  }
  for (int k = 0; k < nreq; ++k) {
    const int b = k & 1, nb = (k + 1) & 1;
    if (!u_out_host[k]) PDE_FAIL("null output buffer");
    if (k + 1 < nreq) {
      if (!u_in_host[k + 1]) PDE_FAIL("null input buffer");
      if (k >= 1) CUDA_OK(cudaStreamWaitEvent(q.h2d, q.in_free[nb], 0));
      CUDA_OK(cudaMemcpyAsync(q.in[nb], u_in_host[k + 1], bytes, cudaMemcpyHostToDevice, q.h2d));
      CUDA_OK(cudaEventRecord(q.in_ready[nb], q.h2d));
    }
    CUDA_OK(cudaStreamWaitEvent(c->stream, q.in_ready[b], 0));
    PDE_OK(launch_unpack(c, s->g, 1, q.in[b], s->u.p, 0));
    CUDA_OK(cudaEventRecord(q.in_free[b], c->stream));
    PDE_OK(launch_apply_bc_values(c, s->g, s->bc, s->u.p));
    PDE_OK(heat_one_solve(s, &st));
    PDE_OK(pipe_push_snapshot(s, u_out_host[k]));
  }
  PDE_OK(pipe_drain(s));
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  st.solve_ms = ms;
  st.setup_ms = s->setup_ms;
  st.launches = c->launches - l0;
  if (st_out) *st_out = st;
  return 0;
}

extern "C" int pde_heat_solve(pde_ctx* c, const pde_heat_params* p, const pde_solver_opts* o, const double* u0,
                              double* values_out, double* times_out, pde_stats* st_out) {
  if (!values_out || !times_out) PDE_FAIL("null output buffers");
  pde_heat_state* s = nullptr;
  PDE_OK(pde_heat_open(c, p, o, &s));
  int rc = 0;
  pde_stats acc;
  stats_init(&acc, (long long)s->g.nn[0] * s->g.nn[1] * s->g.nzg);
  do {
    if (p->initial_type == PDE_IC_ARRAY) {
      if (!u0) { pde_set_error("initial_type array needs u0"); rc = 1; break; }
      if ((rc = pde_heat_set_state(s, u0))) break;
    }
    long long snap = 0;
    if (p->steady) {
      pde_stats st;
      if ((rc = pde_heat_step(s, 1, &st))) break;
      acc = st;
      if ((rc = pde_heat_get_state(s, values_out))) break;
      times_out[0] = 0.0;
      break;
    }
    // snapshots leave through the copy pipeline: the D2H of snapshot k overlaps step k+1 (fully when values_out
    // is pinned host memory; a pageable destination makes the copy call itself blocking, which is still correct)
    if ((rc = pipe_init(s, false))) break;
    s->pipe.nout = 0;
    if ((rc = pipe_push_snapshot(s, values_out))) break;
    times_out[snap++] = 0.0;
    const int stride = p->snapshot_stride > 0 ? p->snapshot_stride : 1;
    const int verify = s->o.verify_residual;
    for (int step = 0; step < p->num_steps; ++step) {
      pde_stats st;
      s->o.verify_residual = step == p->num_steps - 1 ? verify : -1;   // true residual of the LAST step only
      if ((rc = pde_heat_step(s, 1, &st))) break;
      acc.true_relres = st.true_relres;
      acc.iters_total += st.iters_total;
      acc.precond_applies += st.precond_applies;
      acc.solves += st.solves;
      acc.converged &= st.converged;
      acc.levels = st.levels;
      acc.final_relres = st.final_relres;
      acc.solve_ms += st.solve_ms;
      acc.launches += st.launches;
      if ((step + 1) % stride == 0) {
        if ((rc = pipe_push_snapshot(s, values_out + snap * s->nloc))) break;
        times_out[snap++] = (step + 1) * p->dt;
      }
    }
    if (!rc) rc = pipe_drain(s);
    acc.setup_ms = s->setup_ms;
  } while (0);
  pde_heat_close(s);
  if (st_out) *st_out = acc;
  return rc;
}

// ---- generic operator entry points -------------------------------------------------------------------
static int setup_op(pde_ctx* c, const pde_op_params* p, Operator* A, int* ncomp) {
  Grid g;
  PDE_OK(make_grid(p->dim, p->n, p->L, c->rank, c->world, &g));
  BcDev bc;
  PDE_OK(make_bc(p->dim, p->n, &p->bc, &bc));
  if (p->kind == PDE_OP_ELASTICITY) {
    if (p->dim < 2) PDE_FAIL("elasticity operator needs dim 2 or 3");
    PDE_OK(A->setup_elasticity(c, g, bc, p->lam, p->mu));
  } else {
    double a = p->kind == PDE_OP_MASS ? 1.0 : (p->kind == PDE_OP_STIFFNESS ? 0.0 : p->alpha);
    double b = p->kind == PDE_OP_MASS ? 0.0 : (p->kind == PDE_OP_STIFFNESS ? 1.0 : p->beta);
    PDE_OK(A->setup_scalar(c, g, bc, a, b));
  }
  *ncomp = A->tab.ncomp;
  return 0;
}

struct OpGuard {
  Operator A;
  Field x, y, r;
  PcgWork w;
  Hierarchy mg;
  ~OpGuard() { A.release(); x.release(); y.release(); r.release(); w.release(); mg.release(); }
};

// CUDA devices visible to this process; 0 (not an error) without a driver or a GPU
extern "C" int pde_device_count(int32_t* count) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); n = 0; }
  if (count) *count = n;
  return 0;
}

extern "C" int pde_op_apply(pde_ctx* c, const pde_op_params* p, const double* x, double* y) {
  if (!c || !p || !x || !y) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(c->device));
  OpGuard G;
  int nc;
  PDE_OK(setup_op(c, p, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(G.x.alloc(c, g, nc));
  PDE_OK(G.y.alloc(c, g, nc));
  const long long nloc = (long long)g.nn[0] * g.nn[1] * g.nzl;
  DevMem dense;
  PDE_OK(dense.alloc(sizeof(double) * nloc * nc));
  PDE_OK(h2d(c, dense.p, x, sizeof(double) * nloc * nc));
  PDE_OK(launch_unpack(c, g, nc, (const double*)dense.p, G.x.p, 0));
  StencilArgs a;
  a.x = G.x.p; a.y = G.y.p; a.variant = p->variant; a.reduce_slot_xy = S_XY;
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, G.x.p));
  PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  PDE_OK(launch_pack(c, g, nc, G.y.p, (double*)dense.p, 0));
  return d2h(c, y, dense.p, sizeof(double) * nloc * nc);
}

extern "C" int pde_op_bench(pde_ctx* c, const pde_op_params* p, int reps, int warmup, double* ms_per_apply,
                            int64_t* ndofs) {
  if (!c || !p) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(c->device));
  OpGuard G;
  int nc;
  PDE_OK(setup_op(c, p, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(G.x.alloc(c, g, nc));
  PDE_OK(G.y.alloc(c, g, nc));
  PDE_OK(launch_fill_pattern(c, g, G.A.bc, nc, G.x.p));
  StencilArgs a;
  a.x = G.x.p; a.y = G.y.p; a.variant = p->variant; a.reduce_slot_xy = S_XY;
  for (int i = 0; i < warmup; ++i) PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  for (int i = 0; i < reps; ++i) PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  if (ms_per_apply) *ms_per_apply = ms / (reps > 0 ? reps : 1);
  if (ndofs) *ndofs = (int64_t)g.nn[0] * g.nn[1] * g.nzl * nc;
  return 0;
}

// One smoother / residual kernel of the solver on caller data, so that every mode of the sweep kernels can be checked
// against the generic table kernel (variant 1) and the oracle matrix.
//   mode 0: y = A x            1: y = b - A x          2: Chebyshev restart  y = x + c2 D^-1 (b - A x)
//   mode 3: y = x + c1 (x - xprev) + c2 D^-1 (b - A x), output written over xprev as in the solver
//   mode 4: as 3 with xprev = 0 (prev_mode 2)
//   mode 5: the fused first two sweeps from a zero guess, x1 = c2 D^-1 b, y = x1 + c1 x1 + c2 D^-1 (b - A x1)
//           (uniform-diagonal scalar operators, and the 3-D elasticity operator with its two-layer face kernel)
static int sweep_args(int mode, double c1, double c2, const Field& x, const Field& b, Field& y, StencilArgs* a) {
  if (mode < 0 || mode > 5) PDE_FAIL("sweep mode must be 0..5");
  if (mode == 5) {   // the first two sweeps from a zero guess in one pass: the input field is the right-hand side
    a->x = b.p; a->y = y.p; a->cheby = 2; a->s0 = c2; a->c1 = c1; a->c2 = c2;
    return 0;
  }
  a->x = x.p; a->y = y.p;
  if (mode >= 1) a->b = b.p;
  if (mode == 1) { a->bscale = 1.0; a->ascale = -1.0; }
  if (mode >= 2) { a->cheby = 1; a->c1 = mode == 2 ? 0.0 : c1; a->c2 = c2; }
  if (mode == 3) { a->prev_mode = 1; a->xprev = y.p; }
  if (mode == 4) a->prev_mode = 2;
  return 0;
}

extern "C" int pde_op_sweep(pde_ctx* c, const pde_op_params* p, int mode, double c1, double c2, const double* x,
                            const double* b, const double* xprev, double* y, double* dots) {
  if (!c || !p || !x || !y) PDE_FAIL("null argument");
  if (mode >= 1 && !b) PDE_FAIL("this sweep mode needs b");
  if (mode == 3 && !xprev) PDE_FAIL("sweep mode 3 needs xprev");
  CUDA_OK(cudaSetDevice(c->device));
  OpGuard G;
  Field fb;
  struct Rel { Field* f; ~Rel() { f->release(); } } rel{&fb};
  int nc;
  PDE_OK(setup_op(c, p, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(G.x.alloc(c, g, nc));
  PDE_OK(G.y.alloc(c, g, nc));
  PDE_OK(fb.alloc(c, g, nc));
  const long long nloc = (long long)g.nn[0] * g.nn[1] * g.nzl;
  DevMem dense;
  PDE_OK(dense.alloc(sizeof(double) * nloc * nc));
  auto up = [&](const double* h, double* padded) -> int {
    PDE_OK(h2d(c, dense.p, h, sizeof(double) * nloc * nc));
    return launch_unpack(c, g, nc, (const double*)dense.p, padded, 0);
  };
  PDE_OK(up(x, G.x.p));
  if (mode >= 1) PDE_OK(up(b, fb.p));
  if (mode == 3) PDE_OK(up(xprev, G.y.p));
  StencilArgs a;
  PDE_OK(sweep_args(mode, c1, c2, G.x, fb, G.y, &a));
  a.variant = p->variant;
  a.reduce_slot_xy = mode == 5 ? -1 : S_XY;
  CUDA_OK(cudaMemsetAsync(c->scal + S_XY, 0, 2 * sizeof(double), c->stream));
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, mode == 5 ? fb.p : G.x.p));
  PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  if (dots) PDE_OK(read_scal(c, S_XY, 2, dots));
  PDE_OK(launch_pack(c, g, nc, G.y.p, (double*)dense.p, 0));
  return d2h(c, y, dense.p, sizeof(double) * nloc * nc);
}

// Test entry: the constant right-hand-side term of the stencil kernels (heat source f m, elasticity body force) on
// caller data, y = g (.) m - A x through the same launch_stencil call as the solves
extern "C" int pde_op_load(pde_ctx* c, const pde_op_params* p, const double gconst[3], const double* x, double* y) {
  if (!c || !p || !gconst || !x || !y) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(c->device));
  OpGuard G;
  int nc;
  PDE_OK(setup_op(c, p, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(G.x.alloc(c, g, nc));
  PDE_OK(G.y.alloc(c, g, nc));
  const long long nloc = (long long)g.nn[0] * g.nn[1] * g.nzl;
  DevMem dense;
  PDE_OK(dense.alloc(sizeof(double) * nloc * nc));
  PDE_OK(h2d(c, dense.p, x, sizeof(double) * nloc * nc));
  PDE_OK(launch_unpack(c, g, nc, (const double*)dense.p, G.x.p, 0));
  StencilArgs a;
  a.x = G.x.p; a.y = G.y.p; a.bscale = 1.0; a.ascale = -1.0; a.variant = p->variant; a.reduce_slot_xy = S_XY;
  for (int i = 0; i < nc; ++i) a.bconst[i] = gconst[i];
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, G.x.p));
  PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  PDE_OK(launch_pack(c, g, nc, G.y.p, (double*)dense.p, 0));
  return d2h(c, y, dense.p, sizeof(double) * nloc * nc);
}

// Test entry: the raw P2 load vector of the cosine / sine initial condition on the box [lo, hi] (project_trig_ic's
// right-hand side, before the mass solve)
extern "C" int pde_trig_ic_load(pde_ctx* c, int dim, const int32_t n[3], const double lo[3], const double hi[3],
                                int initial_type, double amplitude, double wavenumber, double* load_out) {
  if (!c || !n || !lo || !hi || !load_out) PDE_FAIL("null argument");
  if (c->world > 1) PDE_FAIL("pde_trig_ic_load runs on one GPU");
  if (dim < 1 || dim > 3) PDE_FAIL("dim must be 1, 2 or 3");
  if (initial_type != PDE_IC_COSINE && initial_type != PDE_IC_SINE) PDE_FAIL("initial_type must be cosine or sine");
  CUDA_OK(cudaSetDevice(c->device));
  double L[3] = {1.0, 1.0, 1.0};
  for (int k = 0; k < dim; ++k) {
    L[k] = hi[k] - lo[k];
    if (!(L[k] > 0)) PDE_FAIL("hi must exceed lo on every axis");
  }
  Grid g;
  PDE_OK(make_grid(dim, n, L, 0, 1, &g));
  Field rhs;
  struct Rel { Field* f; ~Rel() { f->release(); } } rel{&rhs};
  PDE_OK(rhs.alloc(c, g, 1));
  SimplexGeom sg;
  build_simplex_geom(dim, g.h, &sg);
  PDE_OK(launch_p2_load(c, g, sg, amplitude, wavenumber, initial_type == PDE_IC_SINE, n, L, rhs.p, lo));
  const long long nloc = (long long)g.nn[0] * g.nn[1] * g.nzl;
  DevMem dense;
  PDE_OK(dense.alloc(sizeof(double) * nloc));
  PDE_OK(launch_pack(c, g, 1, rhs.p, (double*)dense.p, 0));
  return d2h(c, load_out, dense.p, sizeof(double) * nloc);
}

extern "C" int pde_op_bench_mode(pde_ctx* c, const pde_op_params* p, int mode, int reps, int warmup, double* ms_per_launch,
                                 int64_t* ndofs) {
  if (!c || !p) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(c->device));
  OpGuard G;
  Field fb;
  struct Rel { Field* f; ~Rel() { f->release(); } } rel{&fb};
  int nc;
  PDE_OK(setup_op(c, p, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(G.x.alloc(c, g, nc));
  PDE_OK(G.y.alloc(c, g, nc));
  PDE_OK(fb.alloc(c, g, nc));
  PDE_OK(launch_fill_pattern(c, g, G.A.bc, nc, G.x.p));
  PDE_OK(launch_fill_pattern(c, g, G.A.bc, nc, fb.p));
  StencilArgs a;
  const double lmax = G.A.dev.gershgorin > 0 ? G.A.dev.gershgorin : 2.0;
  PDE_OK(sweep_args(mode, 0.1, 1.0 / lmax, G.x, fb, G.y, &a));
  a.variant = p->variant;
  a.reduce_slot_xy = S_XY;
  for (int i = 0; i < warmup; ++i) PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  for (int i = 0; i < reps; ++i) PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  if (ms_per_launch) *ms_per_launch = ms / (reps > 0 ? reps : 1);
  if (ndofs) *ndofs = (int64_t)g.nn[0] * g.nn[1] * g.nzl * nc;
  return 0;
}

// the GMG hierarchy of the operator solves: levels from the operator, smoother degree and ratio from o
static int build_hierarchy(pde_ctx* c, OpGuard& G, const pde_op_params* p, const pde_solver_opts& o) {
  double p0 = p->kind == PDE_OP_ELASTICITY ? p->lam : (p->kind == PDE_OP_MASS ? 1.0 : (p->kind == PDE_OP_STIFFNESS ? 0.0 : p->alpha));
  double p1 = p->kind == PDE_OP_ELASTICITY ? p->mu : (p->kind == PDE_OP_MASS ? 0.0 : (p->kind == PDE_OP_STIFFNESS ? 1.0 : p->beta));
  PDE_OK(G.mg.build(c, G.A, p->kind == PDE_OP_ELASTICITY ? PDE_OP_ELASTICITY : PDE_OP_HEAT, p0, p1));
  G.mg.nu = o.cheby_degree > 0 ? o.cheby_degree : 2;
  G.mg.ratio = o.cheby_ratio > 1 ? o.cheby_ratio : 8.0;
  return 0;
}

static int solve_with(pde_ctx* c, OpGuard& G, const pde_op_params* p, const pde_solver_opts& o, double* x, double* r,
                      double bn2, pde_stats* st) {
  const int nc = G.A.tab.ncomp;
  long long ndofs = (long long)G.A.g.nn[0] * G.A.g.nn[1] * G.A.g.nzg * nc;
  bool use_mg = false;
  // hierarchy / work-vector setup is timed separately (st->setup_ms); callers subtract it from their region
  cudaEvent_t e0, e1;
  CUDA_OK(cudaEventCreate(&e0));
  CUDA_OK(cudaEventCreate(&e1));
  CUDA_OK(cudaEventRecord(e0, c->stream));
  int rc = 0;
  do {
    if (o.precond != PDE_PRECOND_JACOBI) {
      if ((rc = build_hierarchy(c, G, p, o))) break;
      use_mg = choose_precond(o, c, ndofs, G.mg) == PDE_PRECOND_GMG;
    }
    if ((rc = G.w.alloc(c, G.A.g, nc))) break;
  } while (0);
  cudaEventRecord(e1, c->stream);
  cudaEventSynchronize(e1);
  float sms = 0;
  cudaEventElapsedTime(&sms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (rc) return rc;
  st->setup_ms += sms;
  return pcg_solve(c, G.A, use_mg ? &G.mg : nullptr, G.w, x, r, bn2, o, st);
}

extern "C" int pde_op_solve(pde_ctx* c, const pde_op_params* p, const pde_solver_opts* o_in, const double* b,
                            double* x, pde_stats* st_out) {
  if (!c || !p || !b || !x) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(c->device));
  pde_solver_opts o;
  if (o_in) o = *o_in; else pde_solver_opts_default(&o);
  OpGuard G;
  int nc;
  PDE_OK(setup_op(c, p, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(G.x.alloc(c, g, nc));
  PDE_OK(G.y.alloc(c, g, nc));  // holds b
  PDE_OK(G.r.alloc(c, g, nc));
  const long long nloc = (long long)g.nn[0] * g.nn[1] * g.nzl;
  DevMem dense;
  PDE_OK(dense.alloc(sizeof(double) * nloc * nc));
  PDE_OK(h2d(c, dense.p, b, sizeof(double) * nloc * nc));
  PDE_OK(launch_unpack(c, g, nc, (const double*)dense.p, G.y.p, 0));
  for (int i = 0; i < nc; ++i) PDE_OK(launch_apply_bc_values(c, g, G.A.bc, G.x.p + i * g.comp_stride));
  pde_stats st;
  stats_init(&st, nloc * nc);
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  const long long l0 = c->launches;
  StencilArgs a;
  a.x = G.x.p; a.b = G.y.p; a.y = G.r.p; a.bscale = 1.0; a.ascale = -1.0; a.reduce_slot_xy = S_XY;
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, G.x.p));
  PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_XY, 2));
  double bn2;
  PDE_OK(read_scal(c, S_YY, 1, &bn2));
  PDE_OK(solve_with(c, G, p, o, G.x.p, G.r.p, bn2, &st));
  // true residual
  a.x = G.x.p; a.y = nullptr;
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, G.x.p));
  PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_XY, 2));
  double rr;
  PDE_OK(read_scal(c, S_YY, 1, &rr));
  st.true_relres = bn2 > 0 ? std::sqrt(rr / bn2) : 0.0;
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  st.solve_ms = ms - st.setup_ms;
  st.launches = c->launches - l0;
  PDE_OK(launch_pack(c, g, nc, G.x.p, (double*)dense.p, 0));
  PDE_OK(d2h(c, x, dense.p, sizeof(double) * nloc * nc));
  if (st_out) *st_out = st;
  return 0;
}

// Test entry: the V-cycle of pde_op_solve's GMG path applied ncycles times to one host vector (see the header).  The
// cycles after the first replay the CUDA graph of the levels below level 0 where the hierarchy captures one.
extern "C" int pde_op_vcycle(pde_ctx* c, const pde_op_params* p, const pde_solver_opts* o_in, int32_t ncycles,
                             const double* b, double* z_first, double* z_last, double* bz, pde_mg_info* info) {
  if (!c || !p || !b || !z_first || !z_last || !info) PDE_FAIL("null argument");
  if (ncycles < 1) PDE_FAIL("ncycles must be >= 1");
  if (c->world > 1) PDE_FAIL("pde_op_vcycle runs on one GPU");
  CUDA_OK(cudaSetDevice(c->device));
  pde_solver_opts o;
  if (o_in) o = *o_in; else pde_solver_opts_default(&o);
  OpGuard G;
  int nc;
  PDE_OK(setup_op(c, p, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(G.y.alloc(c, g, nc));  // holds b
  const long long nloc = (long long)g.nn[0] * g.nn[1] * g.nzl;
  const size_t bytes = sizeof(double) * nloc * nc;
  DevMem dense;
  PDE_OK(dense.alloc(bytes));
  PDE_OK(h2d(c, dense.p, b, bytes));
  PDE_OK(launch_unpack(c, g, nc, (const double*)dense.p, G.y.p, 0));
  PDE_OK(build_hierarchy(c, G, p, o));
  const int nl = G.mg.levels();
  if (nl > PDE_MG_MAX_LEVELS) PDE_FAIL("more multigrid levels than pde_mg_info holds");
  for (int k = 0; k < ncycles; ++k) {
    double* z = nullptr;
    bool fused = false;
    PDE_OK(G.mg.vcycle(c, G.A, G.y.p, &z, S_RHO0, &fused));
    if (!fused) PDE_OK(launch_dot(c, g, nc, G.y.p, z, S_RHO0));
    if (k == 0 || k == ncycles - 1) PDE_OK(launch_pack(c, g, nc, z, (double*)dense.p, 0));
    if (k == 0) PDE_OK(d2h(c, z_first, dense.p, bytes));
    if (k == ncycles - 1) PDE_OK(d2h(c, z_last, dense.p, bytes));
  }
  if (bz) PDE_OK(read_scal(c, S_RHO0, 1, bz));
  std::memset(info, 0, sizeof(*info));
  info->levels = nl;
  info->n_dense = G.mg.lv[nl - 1]->n_dense;
  info->graph = G.mg.gstate == 2;
  int ax[3], nax;
  internal_axes(p->dim, ax, &nax);
  for (int l = 0; l < nl; ++l) {
    const MGLevel& L = *G.mg.lv[l];
    for (int q = 0; q < nax; ++q) info->n[l][q] = L.op.g.nc[ax[q]];
    info->lmax[l] = L.op.dev.gershgorin;
    info->paths[l] = L.paths;
  }
  return 0;
}

extern "C" int pde_op_manufactured(pde_ctx* c, const pde_op_params* p, const pde_solver_opts* o_in, double* rel_err,
                                   pde_stats* st_out) {
  if (!c || !p || !rel_err) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(c->device));
  pde_solver_opts o;
  if (o_in) o = *o_in; else pde_solver_opts_default(&o);
  OpGuard G;
  Field ustar;
  struct Rel { Field* f; ~Rel() { f->release(); } } rel{&ustar};
  int nc;
  PDE_OK(setup_op(c, p, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(ustar.alloc(c, g, nc));
  PDE_OK(G.x.alloc(c, g, nc));
  PDE_OK(G.y.alloc(c, g, nc));   // b
  PDE_OK(G.r.alloc(c, g, nc));
  PDE_OK(launch_fill_pattern(c, g, G.A.bc, nc, ustar.p));
  // b = A u*  (also ||b||^2)
  StencilArgs a;
  a.x = ustar.p; a.y = G.y.p; a.reduce_slot_xy = S_XY;
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, ustar.p));
  PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_XY, 2));
  double bn2;
  PDE_OK(read_scal(c, S_YY, 1, &bn2));
  PDE_OK(launch_copy(c, g, nc, G.r.p, G.y.p));   // x0 = 0  =>  r0 = b
  pde_stats st;
  stats_init(&st, (long long)g.nn[0] * g.nn[1] * g.nzg * nc);
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  const long long l0 = c->launches;
  PDE_OK(solve_with(c, G, p, o, G.x.p, G.r.p, bn2, &st));
  // true residual ||b - A x|| / ||b||
  StencilArgs t;
  t.x = G.x.p; t.b = G.y.p; t.y = nullptr; t.bscale = 1.0; t.ascale = -1.0; t.reduce_slot_xy = S_XY;
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, G.x.p));
  PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, t));
  if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_XY, 2));
  double rr;
  PDE_OK(read_scal(c, S_YY, 1, &rr));
  st.true_relres = bn2 > 0 ? std::sqrt(rr / bn2) : 0.0;
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  st.solve_ms = ms - st.setup_ms;
  st.launches = c->launches - l0;
  // error norm: e = x - u*
  PDE_OK(launch_axpy(c, g, nc, G.x.p, ustar.p, -1.0));
  PDE_OK(launch_dot(c, g, nc, G.x.p, G.x.p, S_TMP0));
  PDE_OK(launch_dot(c, g, nc, ustar.p, ustar.p, S_TMP1));
  if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_TMP0, 2));
  double v[2];
  PDE_OK(read_scal(c, S_TMP0, 2, v));
  *rel_err = v[1] > 0 ? std::sqrt(v[0] / v[1]) : 0.0;
  if (st_out) *st_out = st;
  return 0;
}

// ---- elasticity -----------------------------------------------------------------------------------------
// what the elasticity tools solve and project: the operator clamped at x = 0 (1-D: E A u'' on the scalar operator),
// the Lame constants (2-D plane stress or plane strain) and the launch_cell_rhs mode of the projected quantity
// (0 / 1: von Mises stress / strain, 2 / 3: axial strain / stress E u')
struct ElastSetup {
  pde_op_params op;
  double lam = 0.0, mu = 0.0;
  int mode = 0;
};

static int elast_setup(const pde_elast_params* p, ElastSetup* s) {
  if (!(p->E > 0)) PDE_FAIL("E must be > 0");
  const int dim = p->dim;
  if (dim < 1 || dim > 3) PDE_FAIL("dim must be 1, 2 or 3");
  pde_op_params& op = s->op;
  std::memset(&op, 0, sizeof(op));
  op.dim = dim;
  for (int k = 0; k < 3; ++k) { op.n[k] = p->n[k]; op.L[k] = p->L[k]; }
  op.bc.face_on[0] = 1;  // clamp x = 0 (reference :1531-1534, 1681-1684, 1831-1834)
  s->lam = s->mu = 0.0;
  if (dim == 1) {
    op.kind = PDE_OP_HEAT; op.alpha = 0.0; op.beta = p->E * p->area;
  } else {
    if (!(p->nu > -1.0 && p->nu < 0.5)) PDE_FAIL("nu must be in (-1, 0.5)");
    s->mu = p->E / (2.0 * (1.0 + p->nu));
    s->lam = (dim == 2 && p->plane_stress) ? p->E * p->nu / (1.0 - p->nu * p->nu)
                                           : p->E * p->nu / ((1.0 + p->nu) * (1.0 - 2.0 * p->nu));
    op.kind = PDE_OP_ELASTICITY; op.lam = s->lam; op.mu = s->mu;
  }
  s->mode = dim == 1 ? (p->quantity == 1 ? 2 : 3) : (p->quantity == 1 ? 1 : 0);
  return 0;
}

// Test entry: the raw load vector of the projected stress / strain for a caller's displacement (launch_cell_rhs as
// pde_elasticity_solve runs it, before the mass solve)
extern "C" int pde_elast_projection_load(pde_ctx* c, const pde_elast_params* p, const double* disp, double* load_out) {
  if (!c || !p || !disp || !load_out) PDE_FAIL("null argument");
  if (c->world > 1) PDE_FAIL("pde_elast_projection_load runs on one GPU");
  CUDA_OK(cudaSetDevice(c->device));
  ElastSetup es;
  PDE_OK(elast_setup(p, &es));
  const int dim = p->dim, nc = dim == 1 ? 1 : dim;
  Grid g;
  PDE_OK(make_grid(dim, p->n, p->L, 0, 1, &g));
  Field u, rhs;
  struct Rel { Field* a; Field* b; ~Rel() { a->release(); b->release(); } } rel{&u, &rhs};
  PDE_OK(u.alloc(c, g, nc));
  PDE_OK(rhs.alloc(c, g, 1));
  const long long nloc = (long long)g.nn[0] * g.nn[1] * g.nzl;
  DevMem dense;
  PDE_OK(dense.alloc(sizeof(double) * nloc * nc));
  PDE_OK(h2d(c, dense.p, disp, sizeof(double) * nloc * nc));
  PDE_OK(launch_unpack(c, g, nc, (const double*)dense.p, u.p, 1));
  SimplexGeom sg;
  build_simplex_geom(dim, g.h, &sg);
  PDE_OK(launch_cell_rhs(c, g, nc, sg, u.p, rhs.p, es.mode, es.lam, es.mu, p->E));
  PDE_OK(launch_pack(c, g, 1, rhs.p, (double*)dense.p, 0));
  return d2h(c, load_out, dense.p, sizeof(double) * nloc);
}

extern "C" int pde_elasticity_solve(pde_ctx* c, const pde_elast_params* p, const pde_solver_opts* o_in,
                                    double* field_out, double* disp_out, pde_stats* st_out, pde_stats* st_proj_out) {
  if (!c || !p || !field_out) PDE_FAIL("null argument");
  CUDA_OK(cudaSetDevice(c->device));
  pde_solver_opts o;
  if (o_in) o = *o_in; else pde_solver_opts_default(&o);
  ElastSetup es;
  PDE_OK(elast_setup(p, &es));
  const int dim = p->dim;
  const pde_op_params& op = es.op;
  const double lam = es.lam, mu = es.mu;
  OpGuard G;
  int nc;
  PDE_OK(setup_op(c, &op, &G.A, &nc));
  const Grid& g = G.A.g;
  PDE_OK(G.x.alloc(c, g, nc));
  PDE_OK(G.r.alloc(c, g, nc));
  const long long nloc = (long long)g.nn[0] * g.nn[1] * g.nzl;
  pde_stats st;
  stats_init(&st, nloc * nc);
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  const long long l0 = c->launches;
  // load vector b_{i,c} = f_c * integral(phi_i)  (L = dot(b, v) dx, :1528, 1678, 1828); x0 = 0 => r0 = b
  StencilArgs a;
  a.x = G.x.p; a.y = G.r.p; a.bscale = 1.0; a.ascale = -1.0; a.reduce_slot_xy = S_XY;
  for (int i = 0; i < nc; ++i) a.bconst[i] = p->body[i];
  PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, a));
  if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_XY, 2));
  double bn2;
  PDE_OK(read_scal(c, S_YY, 1, &bn2));
  PDE_OK(solve_with(c, G, &op, o, G.x.p, G.r.p, bn2, &st));
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  st.solve_ms = ms - st.setup_ms;
  st.launches = c->launches - l0;
  if (o.verify_residual >= 0) {
    // true residual b - A u of the returned displacement (kappa ~ 5e8 at config 5: do not trust the recurrence)
    StencilArgs t = a;
    if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, G.x.p));
    PDE_OK(launch_stencil(c, g, G.A.bc, G.A.dev, t));
    if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_XY, 2));
    double rr;
    PDE_OK(read_scal(c, S_YY, 1, &rr));
    st.true_relres = bn2 > 0 ? std::sqrt(rr / bn2) : 0.0;
  }
  // projected scalar: M v = sum_cells value_c |c|/(d+1)   (project(eq_expr, Vs), :1541-1546, 1714, 1862)
  SimplexGeom sg;
  build_simplex_geom(dim, g.h, &sg);
  OpGuard P;
  pde_op_params mp = op;
  mp.kind = PDE_OP_MASS;
  std::memset(&mp.bc, 0, sizeof(mp.bc));
  int nc1;
  PDE_OK(setup_op(c, &mp, &P.A, &nc1));
  PDE_OK(P.x.alloc(c, g, 1));
  PDE_OK(P.r.alloc(c, g, 1));
  pde_stats sp;
  stats_init(&sp, nloc);
  CUDA_OK(cudaEventRecord(c->ev0, c->stream));
  const long long l1 = c->launches;
  if (c->world > 1) PDE_OK(comm_halo_exchange(c, g, nc, G.x.p));
  PDE_OK(launch_cell_rhs(c, g, nc, sg, G.x.p, P.r.p, es.mode, lam, mu, p->E));
  PDE_OK(launch_dot(c, g, 1, P.r.p, P.r.p, S_TMP0));
  if (c->world > 1) PDE_OK(comm_allreduce_scal(c, S_TMP0, 1));
  double pn2;
  PDE_OK(read_scal(c, S_TMP0, 1, &pn2));
  pde_solver_opts po = o;
  po.precond = PDE_PRECOND_JACOBI;   // consistent mass: kappa(D^-1 M) = O(10), Jacobi-PCG converges in ~20 its
  po.rtol = o.rtol < 1e-12 ? o.rtol : 1e-12;
  PDE_OK(solve_with(c, P, &mp, po, P.x.p, P.r.p, pn2, &sp));
  CUDA_OK(cudaEventRecord(c->ev1, c->stream));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  sp.solve_ms = ms - sp.setup_ms;
  sp.launches = c->launches - l1;
  DevMem dense;
  PDE_OK(dense.alloc(sizeof(double) * nloc * nc));
  PDE_OK(launch_pack(c, g, 1, P.x.p, (double*)dense.p, 0));
  PDE_OK(d2h(c, field_out, dense.p, sizeof(double) * nloc));
  if (disp_out) {
    PDE_OK(launch_pack(c, g, nc, G.x.p, (double*)dense.p, 1));
    PDE_OK(d2h(c, disp_out, dense.p, sizeof(double) * nloc * nc));
  }
  if (st_out) *st_out = st;
  if (st_proj_out) *st_proj_out = sp;
  return 0;
}
