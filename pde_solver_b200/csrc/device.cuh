// Device-side helpers and the execution context shared by kernels.cu / solver.cu / cabi.cu.
#pragma once
#include "common.h"

#define RED_MAX_BLOCKS 65536
#define RED_MAX_VALS 4

// scalar slots (device doubles) used by the PCG recurrences
enum { S_RHO0 = 0, S_RHO1 = 1, S_PAP = 2, S_RR = 3, S_XY = 4, S_YY = 5, S_TMP0 = 6, S_TMP1 = 7, S_NSLOTS = 16 };

struct ReduceBuf {
  double* partials;   // [RED_MAX_BLOCKS][RED_MAX_VALS]
  unsigned* counter;  // zero between kernels
};

struct NcclApi;  // comm.cu

struct pde_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_poll = nullptr;
  ReduceBuf red{};
  void* scratch = nullptr;           // grow-only device scratch (cell sums of the von Mises load vector)
  size_t scratch_bytes = 0;
  double* face_partials = nullptr;   // [RED_MAX_BLOCKS][RED_MAX_VALS]: block sums of a deferred face-row kernel
  double* scal = nullptr;     // device [S_NSLOTS]
  double* h_scal = nullptr;   // pinned, mapped host mirror [S_NSLOTS]
  double* h_scal_dev = nullptr;  // device-side address of h_scal
  long long launches = 0;
  // multi-GPU
  int rank = 0, world = 1;
  void* nccl_comm = nullptr;
  NcclApi* nccl = nullptr;
  void* p2p = nullptr;        // peer-memory halo mailboxes (comm.cu), null until the first exchange
  long long n_halo = 0, n_allreduce = 0;   // exchanges / all-reduces issued so far (pde_comm_info)
};

// ---- geometry helpers -----------------------------------------------------------------
__host__ __device__ __forceinline__ int axis_class(int i, int n) {
  return n == 1 ? 1 : (i == 0 ? 0 : (i == n - 1 ? 2 : 1));
}
__host__ __device__ __forceinline__ int node_class(const Grid& g, int ix, int iy, int gz) {
  return axis_class(ix, g.nn[0]) + 3 * axis_class(iy, g.nn[1]) + 9 * axis_class(gz, g.nzg);
}
// Topological DirichletBC of the reference restated on lattice indices (SURVEY A.4):
// x faces first (left/right), then the remaining faces; "other_faces" skips the x-end columns.
__host__ __device__ __forceinline__ bool bc_node(const Grid& g, const BcDev& bc, int ix, int iy, int gz,
                                                 double* val) {
  const bool x0 = g.nc[0] > 0 && ix == 0, x1 = g.nc[0] > 0 && ix == g.nn[0] - 1;
  if (x0 && bc.on[0]) { *val = bc.val[0]; return true; }
  if (x1 && bc.on[1]) { *val = bc.val[1]; return true; }
  if (bc.side_excl && (x0 || x1)) return false;
  if (g.nc[1] > 0) {
    if (iy == 0 && bc.on[2]) { *val = bc.val[2]; return true; }
    if (iy == g.nn[1] - 1 && bc.on[3]) { *val = bc.val[3]; return true; }
  }
  if (g.nc[2] > 0) {
    if (gz == 0 && bc.on[4]) { *val = bc.val[4]; return true; }
    if (gz == g.nzg - 1 && bc.on[5]) { *val = bc.val[5]; return true; }
  }
  return false;
}

// flat offset of Kuhn-stencil neighbour k (folds to a constant after unrolling)
__device__ __forceinline__ long long kOffDdev(int k, int PX, long long plane) {
  constexpr int D[PDE_NOFF][3] = {{0, 0, 0},  {1, 0, 0},  {-1, 0, 0},  {0, 1, 0},  {0, -1, 0},
                                  {0, 0, 1},  {0, 0, -1}, {1, 1, 0},   {-1, -1, 0}, {1, 0, 1},
                                  {-1, 0, -1}, {0, 1, 1}, {0, -1, -1}, {1, 1, 1},   {-1, -1, -1}};
  return D[k][0] + (long long)PX * D[k][1] + plane * D[k][2];
}

// component `ax` of Kuhn-stencil offset k (folds to a constant after unrolling)
__device__ __forceinline__ int kOffDcomp(int k, int ax) {
  constexpr int D[PDE_NOFF][3] = {{0, 0, 0},  {1, 0, 0},  {-1, 0, 0},  {0, 1, 0},  {0, -1, 0},
                                  {0, 0, 1},  {0, 0, -1}, {1, 1, 0},   {-1, -1, 0}, {1, 0, 1},
                                  {-1, 0, -1}, {0, 1, 1}, {0, -1, -1}, {1, 1, 1},   {-1, -1, -1}};
  return D[k][ax];
}

// ----------------------------------------------------------------------------------------------
// deterministic two-stage reduction: per-block partials, last block sums them in fixed order
// ----------------------------------------------------------------------------------------------
#ifdef __CUDACC__
// extra / nextra: partial sums [nextra][RED_MAX_VALS] left by an EARLIER kernel (the deferred face-row kernel), added
// by the last block in fixed order
template <int NV, bool ACC = false>
__device__ __forceinline__ void block_reduce_finalize(double (&v)[NV], ReduceBuf red, double* out,
                                                      const double* extra = nullptr, int nextra = 0) {
  __shared__ double sm[NV][32];
  __shared__ bool is_last;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nth = blockDim.x * blockDim.y;
  const int lane = tid & 31, warp = tid >> 5, nwarp = (nth + 31) >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double s = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) sm[i][warp] = s;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double s = lane < nwarp ? sm[i][lane] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
      if (lane == 0) red.partials[(size_t)blockIdx.x * RED_MAX_VALS + i] = s;
    }
    if (lane == 0) {
      __threadfence();
      unsigned t = atomicAdd(red.counter, 1u);
      is_last = (t == gridDim.x - 1);
    }
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double s = 0.0;
    for (unsigned b = tid; b < gridDim.x; b += nth) s += red.partials[(size_t)b * RED_MAX_VALS + i];
    for (int b = tid; b < nextra; b += nth) s += extra[(size_t)b * RED_MAX_VALS + i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    __syncthreads();
    if (lane == 0) sm[i][warp] = s;
    __syncthreads();
    if (warp == 0) {
      double t = lane < nwarp ? sm[i][lane] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
      if (lane == 0) out[i] = ACC ? out[i] + t : t;
    }
  }
  if (tid == 0) *red.counter = 0u;
}

#endif  // __CUDACC__

// ---- launch geometry for row-structured kernels -----------------------------------------
struct RowLaunch {
  dim3 block, grid;
};
static inline RowLaunch row_launch(const pde_ctx* c, const Grid& g) {
  RowLaunch r;
  int bx = g.nn[0] >= 96 ? 128 : (g.nn[0] > 32 ? 64 : 32);
  int by = 128 / bx;
  long long rows = (long long)g.nn[1] * g.nzl;
  long long blocks = (rows + by - 1) / by;
  long long cap = (long long)c->sm_count * 16;
  if (cap > RED_MAX_BLOCKS) cap = RED_MAX_BLOCKS;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  r.block = dim3(bx, by, 1);
  r.grid = dim3((unsigned)blocks, 1, 1);
  return r;
}
// blocking host <-> device copies on the context's stream
static inline int d2h(pde_ctx* c, void* dst, const void* src, size_t bytes) {
  CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}
static inline int h2d(pde_ctx* c, void* dst, const void* src, size_t bytes) {
  CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

static inline int flat_blocks(const pde_ctx* c, long long n_items, int threads) {
  long long blocks = (n_items + threads - 1) / threads;
  long long cap = (long long)c->sm_count * 8;
  if (cap > RED_MAX_BLOCKS) cap = RED_MAX_BLOCKS;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// ---- kernels.cu API (all asynchronous on ctx->stream) ------------------------------------
struct OpDev {
  int ncomp = 1;
  double* coef = nullptr;   // [27][15][nc*nc]
  double* dinv = nullptr;   // [27][nc]
  double* load = nullptr;   // [27]
  double h_int[PDE_NOFF * 9];  // interior class coefficients (host copy, passed as kernel params)
  double h_dinv_int[3] = {0, 0, 0};  // interior class Jacobi diagonal inverse
  double h_load_int = 0;             // interior class load (integral of the hat function)
  double gershgorin = 0;
  int uniform_diag = 0;  // every free node has the interior-class diagonal (all faces Dirichlet)
};

struct StencilArgs {
  const double* x = nullptr;   // input field (ghost/pad zero)
  const double* b = nullptr;   // optional right-hand side field; if null, B_i = bconst[c]*load[class]
  double* y = nullptr;         // output (may be null: reductions only)
  const double* xprev = nullptr;  // cheby: previous iterate x_{k-1} (may alias y); the direction is never stored,
                                  // d_{k-1} = x_k - x_{k-1}
  int prev_mode = 0;           // 0: restart (c1 = 0), 1: xprev pointer, 2: x_{k-1} = 0, 3: x_{k-1} = s0*dinv*b
  double bconst[3] = {0, 0, 0};
  double bscale = 0, ascale = 1;  // y = bscale*B + ascale*(A x)
  double c1 = 0, c2 = 0;          // cheby: d = c1*(x - xprev) + c2*dinv*(B - A x); y = x + d
  double s0 = 0;                  // cheby == 2: coefficient of the (implicit) first sweep, d1 = s0*dinv*b
  int cheby = 0;                  // 1: one sweep; 2: first TWO sweeps from a zero guess, x = right-hand side
                                  // reduce_slot_xy with cheby: receives sum B.y (one value)
  int reduce_slot_xy = -1;        // scal slot receiving sum x.y (and +1: sum y.y) ; -1: none
  int ghost_out = 0;              // slabs: also compute the ghost planes z = -1 and z = nzl of y (uniform-diagonal
                                  // operators on the sweep kernel only; needs 2 halo planes of x, 1 of b; no reductions)
  int skip_yy = 0;                // the y.y reduction is not needed (PCG only uses x.y = p.Ap)
  int variant = 0;
};

int launch_stencil(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a);
bool sweep_applicable(const Grid& g, int ncomp);
// two restart Chebyshev sweeps in one pass (temporal blocking); *handled = false if not applicable
int launch_post2(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const double* x0, const double* b,
                 double* y, double c2_0, double c1_1, double c2_1, int dot_slot, bool* handled);
// rows of the non-Dirichlet nodes on the domain faces (class-table stencil); reductions are ADDED to the slot
// defer_blocks != nullptr: the kernel only leaves its block sums in c->face_partials (*defer_blocks of them); the
// sweep kernel launched AFTER it adds them in its own finalize (no fence / atomic ticket per face block)
int launch_face_rows(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a,
                     int* defer_blocks = nullptr);
// Jacobi-PCG fused update: x += a p, r -= a q, rho_new = r.dinv r, rr = r.r  (a = rho/pAp from scal)
int launch_cg_update(pde_ctx* c, const Grid& g, const OpDev& op, double* x, double* r, const double* p,
                     const double* q, int slot_rho, int slot_pap, int slot_rho_new, int slot_rr, int jacobi);
// p = z + beta p with z = dinv r (jacobi) or z given; beta = rho_new/rho (first: beta = 0)
int launch_cg_pupdate(pde_ctx* c, const Grid& g, const OpDev& op, double* p, const double* r_or_z,
                      int slot_rho, int slot_rho_new, int first, int jacobi, double* x_deferred = nullptr, int slot_pap = 0);
int launch_dot(pde_ctx* c, const Grid& g, int ncomp, const double* a, const double* b, int slot);
int launch_zero(pde_ctx* c, const Grid& g, int ncomp, double* a);
int launch_copy(pde_ctx* c, const Grid& g, int ncomp, double* dst, const double* src);
int launch_axpy(pde_ctx* c, const Grid& g, int ncomp, double* y, const double* x, double alpha);
// e = u - uold ; uold = u ; u = u + e
int launch_extrapolate(pde_ctx* c, const Grid& g, int ncomp, double* u, double* uold, double* e);
// first Chebyshev sweep from a zero guess: x = s*dinv*b
int launch_cheby_first(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const double* b, double* x,
                       double s);
int launch_restrict(pde_ctx* c, const Grid& gf, const Grid& gc, const BcDev& bcc, int ncomp, const double* rf,
                    double* bcoarse);
// ghost > 0: also correct `ghost` ghost planes on each side of the fine slab (coarse ghosts must be valid)
int launch_prolong_add(pde_ctx* c, const Grid& gf, const Grid& gc, const BcDev& bcf, int ncomp, const double* xc,
                       double* xf, int ghost = 0);
// fields
int launch_fill_ic(pde_ctx* c, const Grid& g, const BcDev& bc, double* u, double value, int apply_bc);
int launch_halo_verify(pde_ctx* c, const Grid& g, int ncomp, int depth, const double* x, double scale,
                       unsigned long long* bad);
int launch_fill_pattern(pde_ctx* c, const Grid& g, const BcDev& bc, int ncomp, double* x);
int launch_apply_bc_values(pde_ctx* c, const Grid& g, const BcDev& bc, double* u);
int launch_pack(pde_ctx* c, const Grid& g, int ncomp, const double* padded, double* dense, int interleave);
int launch_unpack(pde_ctx* c, const Grid& g, int ncomp, const double* dense, double* padded, int interleave);
int launch_cell_rhs(pde_ctx* c, const Grid& g, int ncomp, const SimplexGeom& sg, const double* u, double* rhs,
                    int mode, double lam, double mu, double Emod);
// load vector of project(A*trig(k x)*trig(k y)*trig(k z) interpolated into P2, V)
int launch_p2_load(pde_ctx* c, const Grid& g, const SimplexGeom& sg, double amp, double kw, int use_sin,
                   const int32_t n_user[3], const double L_user[3], double* rhs, const double* lo_user = nullptr);
int launch_dense_solve(pde_ctx* c, int n, const double* Ainv, const long long* idx, const double* b, double* x);
// multi-rank coarse solve: idx[j] < 0 marks dofs owned by another rank
int launch_dense_gather(pde_ctx* c, int n, const long long* idx, const double* b, double* bglob);
int launch_dense_solve_owned(pde_ctx* c, int n, const double* Ainv, const long long* idx, const double* bglob, double* x);
// mesh
int launch_mesh_coords(pde_ctx* c, int dim, const int32_t n[3], const double L[3], double* out);
int launch_mesh_coords_box(pde_ctx* c, int dim, const int32_t n[3], const double lo[3], const double hi[3], double* out);
int launch_mesh_cells(pde_ctx* c, int dim, const int32_t n[3], int sorted, int ncomp, int layout, int32_t* out);
int launch_bc_mask(pde_ctx* c, const Grid& g, const BcDev& bc, uint8_t* mask, double* vals);

// comm.cu
int comm_allreduce_scal(pde_ctx* c, int slot, int count);
// exchange `depth` (<= PDE_NG) boundary planes with the z-neighbours into the ghost planes
int comm_halo_exchange(pde_ctx* c, const Grid& g, int ncomp, double* field, int depth = 1);
int comm_allreduce_buf(pde_ctx* c, double* buf, size_t count);
int comm_check_error(pde_ctx* c);   // fails if a peer-memory halo wait timed out
