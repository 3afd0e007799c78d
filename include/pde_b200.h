/*
 * pde_b200.h — C ABI of the B200-native structured-mesh P1 solver (libpde_b200.so).
 *
 * This is the drop-in boundary below the Python host layer.  Each entry point names the
 * reference interface it replaces (file:line under /root/reference/fenics_mcp_server.py;
 * the arithmetic itself lives in DOLFIN 2019.1.0 + PETSc, which the reference calls there).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; pde_last_error() gives the
 *     thread-local message.  Nothing is ever printed to stdout (the MCP server owns it).
 *   - the caller owns all host buffers; the library owns device memory behind pde_ctx.
 *   - plain pointers and sizes only; no callbacks; FP64 everywhere; indices int32 unless
 *     stated (global offsets int64).
 *   - dof order of every exported array is the NATURAL lattice order (vertex id =
 *     iz*(nx+1)*(ny+1) + iy*(nx+1) + ix), i.e. DOLFIN with reorder_dofs_serial=False.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef PDE_B200_H
#define PDE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pde_ctx pde_ctx;

/* ---- context / errors ------------------------------------------------------------- */
const char* pde_last_error(void);
int pde_version(void);
/* CUDA devices visible to this process (0 without a GPU; never fails): the tool layer checks PDE_B200_GPUS against it */
int pde_device_count(int32_t* count);
/* one context per GPU (one process per GPU under torchrun; a process may hold several) */
int pde_ctx_create(int device, pde_ctx** out);
int pde_ctx_destroy(pde_ctx* ctx);
/* number of kernels launched through this context since creation (bench "gpu_launches") */
int64_t pde_ctx_launch_count(pde_ctx* ctx);
int pde_ctx_sync(pde_ctx* ctx);
/* CUDA-event timer on the context's compute stream */
int pde_timer_start(pde_ctx* ctx);
int pde_timer_stop(pde_ctx* ctx, double* elapsed_ms);

/* pinned host memory for the host<->device legs of a step (cudaHostAlloc / cudaFreeHost) */
int pde_host_alloc(uint64_t bytes, void** out);
int pde_host_free(void* p);

/* ---- multi-GPU: slab partition along the slowest axis, NCCL over NVLink ------------- */
/* libnccl.so.2 is dlopen()ed from `libnccl_path` (NULL: default search path). */
int pde_nccl_unique_id(const char* libnccl_path, void* id128 /* 128 bytes out */);
int pde_comm_init(pde_ctx* ctx, int rank, int world, const void* id128, const char* libnccl_path);

/* host-only: the slab of vertex planes rank `rank` of `world` owns on multigrid level `level` (0 = the
 * mesh itself, each level halves every axis).  Planes are indexed along the slowest axis of the natural
 * numbering; rank r owns [z0, z0+nzl) of nzg planes.  Returns non-zero if the level does not exist. */
int pde_slab_partition(int dim, const int32_t n[3], int rank, int world, int level, int32_t* z0, int32_t* nzl,
                       int32_t* nzg);

/* time `reps` halo exchanges (one plane each way per z-neighbour, `ncomp` components) of the slab of a
 * dim-D mesh; returns mean ms per exchange and the bytes this rank sends per exchange */
int pde_halo_bench(pde_ctx* ctx, int dim, const int32_t n[3], int ncomp, int reps, double* ms_per_exchange,
                   int64_t* bytes_sent);
/* what the multi-GPU layer does on this context: halo_path 0 = no exchange yet / single GPU, 1 = NCCL send/recv,
 * 2 = peer-memory mailbox kernel over NVLink; counts of halo exchanges and all-reduces issued so far */
int pde_comm_info(pde_ctx* ctx, int32_t* halo_path, int64_t* halo_exchanges, int64_t* allreduces);
/* self-check of the halo exchange (peer-memory kernel or NCCL): `reps` exchanges of `depth` planes of a field
 * defined by the global node index; *mismatches = ghost entries that differ bitwise from the owner's values */
int pde_halo_check(pde_ctx* ctx, int dim, const int32_t n[3], int ncomp, int depth, int reps, int64_t* mismatches);

/* ---- meshes, dof maps, boundary sets (bit-exact rows a2-a4 of SURVEY §8) ------------- */
/* IntervalMesh :229,1516 / RectangleMesh :369,1648 / BoxMesh :533,1803.
 * dim in {1,2,3}; n[k] cells along axis k; domain [0,L[k]].  Generated on the GPU. */
int pde_mesh_counts(int dim, const int32_t n[3], int64_t* nverts, int64_t* ncells);
int pde_mesh_coords(pde_ctx* ctx, int dim, const int32_t n[3], const double L[3],
                    double* coords /* [nverts][dim] */);
/* same generators on [lo, hi] (IntervalMesh(n,a,b) :804,960; RectangleMesh(Point(a,..),..) :1096,1223;
 * BoxMesh(Point(a,..),..) :1360) - the coordinate spaces of the curvilinear tools */
int pde_mesh_coords_box(pde_ctx* ctx, int dim, const int32_t n[3], const double lo[3], const double hi[3],
                        double* coords /* [nverts][dim] */);
/* sorted=0: generation order of each cell's vertices; sorted=1: after mesh.order() */
int pde_mesh_cells(pde_ctx* ctx, int dim, const int32_t n[3], int sorted,
                   int32_t* cells /* [ncells][dim+1] */);
/* FunctionSpace(mesh,"P",1) :230,370,535 (ncomp=1) / VectorFunctionSpace :1649,1804.
 * layout 0: blocked (c*nverts+v, UFC numbering); 1: interleaved (ncomp*v+c). */
int pde_dofmap_cells(pde_ctx* ctx, int dim, const int32_t n[3], int ncomp, int layout,
                     int32_t* cell_dofs /* [ncells][ncomp*(dim+1)] */);

/* Dirichlet specification = the reference's DirichletBC lists.
 * face order: x=0, x=L, then the remaining faces of the present axes (y=0,y=L,z=0,z=L). */
typedef struct pde_bc {
  int32_t face_on[6];
  double face_val[6];
  int32_t side_excludes_xends; /* other_faces predicate :613-616: side faces skip ix=0 / ix=nx */
} pde_bc;
/* mask[v] = 1 where vertex v carries a Dirichlet value; vals[v] its value (0 elsewhere) */
int pde_boundary_mask(pde_ctx* ctx, int dim, const int32_t n[3], const pde_bc* bc,
                      uint8_t* mask /* [nverts] */, double* vals /* [nverts] or NULL */);

/* ---- solver controls ------------------------------------------------------------------ */
enum { PDE_PRECOND_JACOBI = 0, PDE_PRECOND_GMG = 1, PDE_PRECOND_AUTO = 2 };

typedef struct pde_solver_opts {
  double rtol;          /* ||r|| <= rtol*||b||; reference = direct LU, north-star rtol 1e-10 */
  int32_t max_iters;
  int32_t precond;      /* PDE_PRECOND_* */
  int32_t cheby_degree; /* GMG smoother sweeps per side (default 2) */
  int32_t check_every;  /* host convergence poll interval in iterations */
  double cheby_ratio;   /* smoothing interval [lmax/ratio, lmax] */
  int32_t verify_residual; /* 0: recompute ||b - A x||/||b|| after the last solve of a call (pde_stats.true_relres); -1: off */
  int32_t reserved[3];
} pde_solver_opts;
void pde_solver_opts_default(pde_solver_opts* o);

typedef struct pde_stats {
  int64_t ndofs;         /* global dofs of the linear system(s) */
  int64_t iters_total;   /* PCG iterations over all solves of the call */
  int32_t solves;        /* linear solves performed */
  int32_t converged;     /* 1 if every solve reached rtol */
  int32_t levels;        /* multigrid levels used (1 = Jacobi) */
  int32_t precond_applies; /* multigrid preconditioner applications (V-cycles) over all solves of the call: one per
                              PCG iteration (iters_total), none for a start that already meets rtol; 0 for Jacobi */
  double final_relres;   /* last solve: ||r||/||b|| (recurrence) */
  double true_relres;    /* last solve: ||b - A x||/||b|| recomputed */
  double solve_ms;       /* device time of the solver region (CUDA events) */
  double setup_ms;
  int64_t launches;      /* kernels launched by this call */
} pde_stats;

/* ---- heat: _solve_heat_{1,2,3}d_raw :204-338, 345-468, 475-762 (box, uniform kappa) ---- */
enum { PDE_IC_CONSTANT = 0, PDE_IC_ZERO = 1, PDE_IC_COSINE = 2, PDE_IC_SINE = 3, PDE_IC_ARRAY = 4 };

typedef struct pde_heat_params {
  int32_t dim;
  int32_t n[3];
  double L[3];
  double diffusivity;
  double dt;
  int32_t num_steps;
  int32_t steady;
  double source_value;       /* 0 when source_type == "none" */
  int32_t initial_type;      /* PDE_IC_* */
  int32_t snapshot_stride;   /* keep every k-th step (1 = the reference's behaviour) */
  double T_initial;
  double initial_amplitude;
  double initial_wavenumber;
  pde_bc bc;
} pde_heat_params;

/* values_out: [nsnap][nverts] natural order, nsnap = 1 + num_steps/stride (steady: 1);
 * times_out: [nsnap]; u0 (PDE_IC_ARRAY only): [nverts] host initial field. */
int pde_heat_solve(pde_ctx* ctx, const pde_heat_params* p, const pde_solver_opts* o,
                   const double* u0, double* values_out, double* times_out, pde_stats* st);

/* resident time stepper (bench / large runs): state stays in HBM between calls */
typedef struct pde_heat_state pde_heat_state;
int pde_heat_open(pde_ctx* ctx, const pde_heat_params* p, const pde_solver_opts* o,
                  pde_heat_state** out);
int pde_heat_set_state(pde_heat_state* s, const double* u_host /* [local nverts] */);
int pde_heat_step(pde_heat_state* s, int nsteps, pde_stats* st);
int pde_heat_get_state(pde_heat_state* s, double* u_host /* [local nverts] */);
/* nreq independent one-step advances u_in[k] -> u_out[k] (each [local nverts], host memory; pinned buffers from
 * pde_host_alloc give full overlap): upload of request k+1 and download of result k-1 run on separate copy streams
 * while request k is solved.  Same arithmetic per request as set_state + step(1) + get_state. */
int pde_heat_advance_batch(pde_heat_state* s, int nreq, const double* const* u_in_host,
                           double* const* u_out_host, pde_stats* st);
int64_t pde_heat_local_nverts(pde_heat_state* s);
int pde_heat_close(pde_heat_state* s);

/* ---- curvilinear heat tools: _solve_heat_{1d,2d}_cylindrical_raw, _solve_heat_{1d,2d,3d}_spherical_raw :769-1464 ----
 * Same backward-Euler / steady P1 solve on the coordinate-space mesh [lo,hi] with ONE scalar weight in every term:
 *   a = w u v dx + dt k w grad(u).grad(v) dx,  L = w u_n v dx + dt w f v dx,
 *   w = x0^weight_rpow * (weight_sin_axis1 ? sin(x1) : 1), an Expression of degree weight_degree (1 or 2).
 * The initial state of the curvilinear tools is the constant T_initial (every initial_type falls back to it);
 * the 3D cylinder / composite-core branches honour initial_type like the box solver.  PDE_IC_ARRAY is refused:
 * a host initial field goes through the resident stepper (pde_wheat_open + pde_wheat_set_state), which also serves
 * runs whose snapshots do not fit in host memory (one pde_wheat_get_state per kept snapshot). */
typedef struct pde_wheat_params {
  int32_t dim;
  int32_t n[3];
  double lo[3], hi[3];
  int32_t weight_rpow;        /* 1: w ~ r (cylindrical), 2: w ~ r^2 (spherical) */
  int32_t weight_sin_axis1;   /* 1: times sin(x[1]) (2D/3D spherical) */
  int32_t weight_degree;      /* degree of the weight Expression: 1 or 2 */
  int32_t steady;
  double diffusivity;
  double dt;
  int32_t num_steps;
  int32_t snapshot_stride;
  double source_value;
  double T_initial;
  pde_bc bc;
  /* cylinder / composite-core branches of _solve_heat_3d_raw (:512-572, 642-645; dim 3 only) */
  int32_t weight_kind;        /* 0: separable weight above; 1: w = sqrt(x1^2 + x2^2) (degree 2), the BoxMesh "cylinder" */
  int32_t has_core;           /* 1: DG0 diffusivity = core_diffusivity on cells with sqrt(x1^2+x2^2) < core_radius */
  double core_radius;
  double core_diffusivity;
  int32_t initial_type;       /* PDE_IC_CONSTANT / PDE_IC_ZERO / PDE_IC_COSINE / PDE_IC_SINE */
  int32_t reserved0;
  double initial_amplitude;
  double initial_wavenumber;
} pde_wheat_params;
/* o->precond: PDE_PRECOND_GMG runs GMG-PCG with Galerkin coarse operators (P^T A P) while every axis halves evenly;
 * st->levels and st->true_relres (||b - A x||/||b|| of the last solve, full assembled stencil) are filled.  A grid
 * with an odd cell count falls back to Jacobi-PCG (levels = 1).  PDE_PRECOND_JACOBI and PDE_PRECOND_AUTO run
 * Jacobi-PCG (true_relres = NaN). */
int pde_wheat_solve(pde_ctx* ctx, const pde_wheat_params* p, const pde_solver_opts* o,
                    double* values_out /* [nsnap][nverts] */, double* times_out, pde_stats* st);
/* resident stepper of the same solve: state stays in HBM between calls, pde_wheat_solve is open + step(1) per step
 * + get_state per kept snapshot.  open assembles, builds the GMG hierarchy (o->precond as above) and sets the
 * initial state from initial_type (num_steps and snapshot_stride are not used).  set_state loads a host field and
 * re-applies the Dirichlet values.  step runs nsteps backward-Euler steps (steady: the one solve, from the current
 * state as starting guess); st covers this call, true_relres its last step.  One GPU only. */
typedef struct pde_wheat_state pde_wheat_state;
int pde_wheat_open(pde_ctx* ctx, const pde_wheat_params* p, const pde_solver_opts* o, pde_wheat_state** out);
int pde_wheat_set_state(pde_wheat_state* s, const double* u_host /* [nverts] natural order */);
int pde_wheat_step(pde_wheat_state* s, int nsteps, pde_stats* st);
int pde_wheat_get_state(pde_wheat_state* s, double* u_host /* [nverts] natural order */);
int64_t pde_wheat_local_nverts(pde_wheat_state* s);
int pde_wheat_close(pde_wheat_state* s);
/* Operator of multigrid level `level` of the GMG path: n_out = cells per user axis of that level (0 for absent axes),
 * coef_out = [nk][nverts] in natural vertex order, nk = 3 / 7 / 15 (1-D / 2-D / 3-D): entry [k][i] = a(i, i + d_k)
 * with d_k the Kuhn offsets in internal axes (x, y, z; 2-D: x, z) in the order {0, +x, -x, +y, -y, +z, -z, +xy, -xy,
 * +xz, -xz, +yz, -yz, +xyz, -xyz} restricted to the present axes.  Rows and columns of Dirichlet vertices are zero.
 * coef_out = NULL only fills n_out.  Non-zero if the level does not exist. */
int pde_wheat_level_coefs(pde_ctx* ctx, const pde_wheat_params* p, int level, int32_t n_out[3], double* coef_out);

/* ---- elasticity: _solve_elasticity_{1,2,3}d_static :1470-1587, 1593-1743, 1749-1892 ---- */
typedef struct pde_elast_params {
  int32_t dim;
  int32_t n[3];
  double L[3];
  double E;
  double nu;
  double body[3];
  int32_t quantity;       /* 0 = stress, 1 = strain */
  int32_t plane_stress;   /* 2D only */
  double area;            /* 1D only */
} pde_elast_params;

/* field_out: [nverts] projected von-Mises (1D: axial) stress/strain, natural order.
 * disp_out: optional [nverts][dim] displacement (never exported by the reference). */
int pde_elasticity_solve(pde_ctx* ctx, const pde_elast_params* p, const pde_solver_opts* o,
                         double* field_out, double* disp_out, pde_stats* st, pde_stats* st_proj);

/* ---- operator-level entry points (parity tests and micro-benchmarks) -------------------- */
enum { PDE_OP_HEAT = 0, PDE_OP_MASS = 1, PDE_OP_STIFFNESS = 2, PDE_OP_ELASTICITY = 3 };

typedef struct pde_op_params {
  int32_t kind;       /* PDE_OP_* */
  int32_t dim;
  int32_t n[3];
  double L[3];
  double alpha;       /* heat: A = alpha*M + beta*K */
  double beta;
  double lam, mu;     /* elasticity */
  pde_bc bc;          /* rows at Dirichlet vertices are masked to zero */
  int32_t variant;    /* 0 = auto (fastest kernel), 1 = generic table kernel */
} pde_op_params;

/* host-only: interior/boundary stencil table [27][15][ncomp*ncomp] (no GPU needed) */
int pde_op_table(const pde_op_params* p, double* table, int32_t* ncomp);
/* y = A x on the device; x,y host arrays [ncomp][nverts] (blocked), natural order */
int pde_op_apply(pde_ctx* ctx, const pde_op_params* p, const double* x, double* y);
/* time `reps` device-resident applications (+fused dot); returns mean ms per apply */
int pde_op_bench(pde_ctx* ctx, const pde_op_params* p, int reps, int warmup, double* ms_per_apply,
                 int64_t* ndofs);
/* one smoother / residual kernel of the solver on host arrays [ncomp][nverts] (test entry: every mode of the
 * specialised sweep kernels against the generic kernel and the oracle matrix).
 *   mode 0: y = A x   1: y = b - A x   2: y = x + c2 D^-1 (b - A x)
 *   mode 3: y = x + c1 (x - xprev) + c2 D^-1 (b - A x)   4: as 3 with xprev = 0
 *   mode 5: the fused first two sweeps from a zero guess: x1 = c2 D^-1 b, y = (1 + c1) x1 + c2 D^-1 (b - A x1)
 * Dirichlet rows: 0 in modes 0/1, x in modes 2..4.  dots (may be NULL) receives the fused reductions
 * (modes 0/1: x.y, y.y; modes 2..4: b.y over free rows, second value unspecified). */
int pde_op_sweep(pde_ctx* ctx, const pde_op_params* p, int32_t mode, double c1, double c2, const double* x,
                 const double* b, const double* xprev, double* y, double* dots);
/* as pde_op_bench for one of the sweep modes above (device-resident pattern data) */
int pde_op_bench_mode(pde_ctx* ctx, const pde_op_params* p, int32_t mode, int32_t reps, int32_t warmup,
                      double* ms_per_launch, int64_t* ndofs);
/* solve A x = b (symmetric Dirichlet elimination) from host arrays; PCG per `o` */
int pde_op_solve(pde_ctx* ctx, const pde_op_params* p, const pde_solver_opts* o, const double* b,
                 double* x, pde_stats* st);

/* Device-resident manufactured-solution check for sizes no CPU oracle can reach (SURVEY §8c iv-c):
 * u*_i = sin(0.37 i + comp) + 0.5 on free nodes (0 on Dirichlet nodes), b = A u* with the matrix-free
 * operator, solve A x = b from x = 0 with the configured PCG, return ||x - u*||_2 / ||u*||_2.
 * Nothing but scalars crosses the host boundary. */
int pde_op_manufactured(pde_ctx* ctx, const pde_op_params* p, const pde_solver_opts* o, double* rel_l2_error,
                        pde_stats* st);

/* ---- multigrid V-cycle test entry points ---------------------------------------------------------------------
 * The V-cycle is a fixed linear map z = B b.  These entries build the hierarchy the solver builds, apply B to a host
 * vector `ncycles` times and return it, so that tests can compare B with a model of it vector by vector. */
#define PDE_MG_MAX_LEVELS 16
/* paths bits: fused kernels a level actually ran (k_sweep / generic FIRST2 pass of the first two pre-smoothing
 * sweeps, k_heat_post2 post-smoothing, k_heat_post2 residual + restriction); bit 4 is unused */
enum { PDE_MG_FIRST2 = 1, PDE_MG_HEAT_POST2 = 2, PDE_MG_RESID_RESTRICT = 8 };
typedef struct pde_mg_info {
  int32_t levels, n_dense;
  int32_t graph;                        /* 1: the last cycle replayed a captured CUDA graph */
  int32_t reserved;
  int32_t n[PDE_MG_MAX_LEVELS][3];      /* cells per user axis of each level (0 for absent axes) */
  double lmax[PDE_MG_MAX_LEVELS];       /* Chebyshev upper bound each level used */
  uint32_t paths[PDE_MG_MAX_LEVELS];    /* PDE_MG_* bits, accumulated over the cycles of the call */
} pde_mg_info;
/* Box operators (heat / elasticity): the hierarchy of pde_op_solve's GMG path (nu and ratio from o, with the same
 * environment overrides), run ncycles >= 1 times on the same b with the fused b.z of the PCG.  This always runs the
 * hierarchy's cycle, a one-level hierarchy included.  b, z_first (cycle 1), z_last (cycle ncycles): host arrays
 * [ncomp][nverts], natural order; bz (may be NULL): the fused b.z of the last cycle (free rows).  One GPU only. */
int pde_op_vcycle(pde_ctx* ctx, const pde_op_params* p, const pde_solver_opts* o, int32_t ncycles, const double* b,
                  double* z_first, double* z_last, double* bz, pde_mg_info* info);
/* The same for the weighted operators of pde_wheat_solve (the steady / backward-Euler matrix of p) and their Galerkin
 * hierarchy; paths stay 0, graph is 0.  Non-zero if the grid does not coarsen (the solve runs Jacobi-PCG then). */
int pde_wheat_vcycle(pde_ctx* ctx, const pde_wheat_params* p, int32_t ncycles, const double* b, double* z_first,
                     double* z_last, double* bz, pde_mg_info* info);

/* ---- load-vector test entry points ------------------------------------------------------------------------------
 * The vectors the solvers build on the device before they solve, returned raw, so that tests can compare them with a
 * reference entry by entry.  Each runs the production launch of its solver on one GPU; natural vertex order. */
/* b_i = sum over the simplices c that contain vertex i of value_c |c| / (dim + 1), value_c the von Mises stress /
 * strain (1-D: E u' / u') of the displacement disp [nverts][dim] (the layout of disp_out), with the clamp, Lame
 * constants and quantity of pde_elasticity_solve.  load_out: [nverts]. */
int pde_elast_projection_load(pde_ctx* ctx, const pde_elast_params* p, const double* disp, double* load_out);
/* the P2 load of the cosine / sine initial condition amplitude * prod_q trig(wavenumber x_q) on the box [lo, hi]
 * (initial_type PDE_IC_COSINE or PDE_IC_SINE): b_i = int I_P2(f) phi_i.  load_out: [nverts]. */
int pde_trig_ic_load(pde_ctx* ctx, int dim, const int32_t n[3], const double lo[3], const double hi[3],
                     int initial_type, double amplitude, double wavenumber, double* load_out);
/* the assembly of pde_wheat_solve: coefA (A = alpha M_w + beta K_w of p, steady: alpha = 0, beta = diffusivity;
 * transient: alpha = 1, beta = dt diffusivity) and coefM (M_w), each [nk][nverts] with both halves of the stencil,
 * nk and the offset order as in pde_wheat_level_coefs; no Dirichlet masking.  load: [nverts], m_i = int I(w) phi_i. */
int pde_wheat_assembly(pde_ctx* ctx, const pde_wheat_params* p, double* coefA, double* coefM, double* load);
/* y = g (.) m - A x with m_i = int phi_i and component c scaled by g[c], Dirichlet rows 0 (the constant term of the
 * heat source and the elasticity body force).  x, y: [ncomp][nverts] blocked. */
int pde_op_load(pde_ctx* ctx, const pde_op_params* p, const double g[3], const double* x, double* y);

#ifdef __cplusplus
}
#endif
#endif /* PDE_B200_H */
