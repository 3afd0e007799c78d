// Galerkin geometric multigrid for the per-node operators of weighted.cu (curvilinear tools, BoxMesh cylinder,
// composite core).  Jacobi-PCG needs O(1/h) iterations on these operators; a V-cycle with Galerkin coarse operators
// keeps the count nearly flat under refinement, and Galerkin (not re-discretisation) keeps the DG0 core boundary of
// the fine grid on every level.
//
// Storage: the operator is symmetric, so each level keeps the centre and ONE coefficient per +/- Kuhn offset pair
// (8 planes in 3-D, 4 in 2-D, 2 in 1-D); a(i, i-k) = a(i-k, i) is read at the neighbour.  Rows and columns of
// Dirichlet nodes are zero, so every level stores exactly its free-free block.
// Coarse operators: P^T A P with P the Kuhn edge-midpoint prolongation of k_prolong_add (R = P^T is k_restrict).
// The P1 spaces are nested, so the product keeps the 15 (7, 3) point pattern; k_wgalerkin counts any entry outside it.
// Smoother: Chebyshev(2)-Jacobi on [lmax/8, lmax], lmax = Gershgorin bound of D^-1 A (k_wlmax); coarsest level:
// dense inverse (<= PDE_DENSE_MAX free nodes) or 8 sweeps at ratio 30.
#include <cmath>
#include <cstring>

#include "wmg.cuh"

enum { W_FIRST = 0, W_APPLY = 1, W_RESID = 2, W_CHEBY = 3 };

// Hot path.  Dirichlet rows are written as 0.
//   W_FIRST: y = c2 b / a_ii                                  (first Chebyshev sweep from a zero guess)
//   W_APPLY: y = A x                     ; sum x.y -> red_out
//   W_RESID: y = b - A x
//   W_CHEBY: y = x + c1 (x - xprev) + c2 (b - A x) / a_ii     (xprev null: x_prev = 0) ; sum b.y -> red_out
// xprev may alias y (the ping-pong buffer holding x_{k-1} receives x_{k+1}); each thread reads it before writing.
// Flat over the nodes: the +/- z and y neighbours of x and of the coefficient planes are re-read from L2.
template <int NH, int MODE>
__global__ void __launch_bounds__(256)
k_wsweep(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc, const __grid_constant__ WStencil ws,
         const double* __restrict__ h, const double* __restrict__ x, const double* __restrict__ b, const double* xprev,
         double* y, double c1, double c2, int do_reduce, ReduceBuf red, double* red_out) {
  const unsigned n0 = (unsigned)g.nn[0], n1 = (unsigned)g.nn[1];
  const unsigned total = n0 * n1 * (unsigned)g.nzl;   // < 2^32 (checked at launch)
  const long long cs = g.comp_stride;
  double acc = 0.0;
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    const unsigned row = t / n0;
    const int ix = (int)(t - row * n0);
    const int iy = (int)(row % n1), lz = (int)(row / n1);
    const long long i = (long long)g.PX * iy + g.plane * lz + ix;
    double bcv;
    if (bc_node(g, bc, ix, iy, lz + g.z0, &bcv)) { y[i] = 0.0; continue; }
    const double d = h[i];
    double out;
    if (MODE == W_FIRST) {
      out = c2 * b[i] / d;
    } else {
      const double xi = x[i];
      double ax = d * xi;
#pragma unroll
      for (int j = 1; j < NH; ++j) {
        const double* hj = h + j * cs;
        const long long o = ws.off[j];
        ax = fma(hj[i], x[i + o], ax);
        ax = fma(hj[i - o], x[i - o], ax);
      }
      if (MODE == W_APPLY) {
        out = ax;
        acc = fma(xi, out, acc);
      } else if (MODE == W_RESID) {
        out = b[i] - ax;
      } else {
        const double bi = b[i];
        const double xp = xprev ? xprev[i] : 0.0;
        out = xi + c1 * (xi - xp) + c2 * (bi - ax) / d;
        acc = fma(bi, out, acc);
      }
    }
    y[i] = out;
  }
  if ((MODE == W_APPLY || MODE == W_CHEBY) && do_reduce) {
    double v[1] = {acc};
    block_reduce_finalize<1>(v, red, red_out);
  }
}

// level 0: symmetric half of the assembled stencil (a(i, i+k) from row i), free-free block only
__global__ void __launch_bounds__(256)
k_wpack(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc, const __grid_constant__ WStencil ws,
        const double* __restrict__ coefA, double* __restrict__ h) {
  const long long total = (long long)g.nn[0] * g.nn[1] * g.nzl;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long row = t / g.nn[0];
    const int ix = (int)(t - row * g.nn[0]);
    const int iy = (int)(row % g.nn[1]), lz = (int)(row / g.nn[1]), gz = lz + g.z0;
    const long long i = (long long)g.PX * iy + g.plane * lz + ix;
    double bcv;
    const bool fi = !bc_node(g, bc, ix, iy, gz, &bcv);
    h[i] = fi ? coefA[i] : 0.0;
    for (int j = 1; j < ws.nh; ++j) {
      const int jx = ix + ws.dx[j], jy = iy + ws.dy[j], jz = gz + ws.dz[j];   // positive offsets
      const bool in = jx < g.nn[0] && jy < g.nn[1] && jz < g.nzg;
      const bool fj = in && !bc_node(g, bc, jx, jy, jz, &bcv);
      h[i + j * g.comp_stride] = fi && fj ? coefA[i + (2 * j - 1) * g.comp_stride] : 0.0;
    }
  }
}

// Coarse row I of P^T A_f P (free-free): fine nodes a = 2I + o_m carry weight 1 (m = 0) or 1/2; each fine entry
// A_f(a, b) is spread onto b's coarse parents ((b - p)/2, (b + p)/2), p = parity of b, 1/2 each (p = 0: b/2, 1).
// Entries landing outside the coarse stencil are counted in *bad (the product is in-pattern for nested P1 spaces).
__global__ void __launch_bounds__(128)
k_wgalerkin(const __grid_constant__ Grid gf, const __grid_constant__ Grid gc, const __grid_constant__ BcDev bc,
            const __grid_constant__ WStencil wsf, const __grid_constant__ WStencil wsc, const double* __restrict__ hf,
            double* __restrict__ hc, int* bad) {
  const long long total = (long long)gc.nn[0] * gc.nn[1] * gc.nzl;
  const bool hy = gc.nc[1] > 0, hz = gc.nc[2] > 0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long row = t / gc.nn[0];
    const int ix = (int)(t - row * gc.nn[0]);
    const int iy = (int)(row % gc.nn[1]), lz = (int)(row / gc.nn[1]);
    const long long ic = (long long)gc.PX * iy + gc.plane * lz + ix;
    double bcv;
    if (bc_node(gc, bc, ix, iy, lz, &bcv)) {
      for (int j = 0; j < wsc.nh; ++j) hc[ic + j * gc.comp_stride] = 0.0;
      continue;
    }
    double acc[PDE_NOFF];
#pragma unroll
    for (int k = 0; k < PDE_NOFF; ++k) acc[k] = 0.0;
    for (int m = 0; m < gf.nk; ++m) {
      const int ax = 2 * ix + gf.kdx[m], ay = 2 * iy + gf.kdy[m], az = 2 * lz + gf.kdz[m];
      if (ax < 0 || ax >= gf.nn[0] || ay < 0 || ay >= gf.nn[1] || az < 0 || az >= gf.nzl) continue;
      const double wm = m == 0 ? 1.0 : 0.5;
      const long long a = (long long)gf.PX * ay + gf.plane * az + ax;
      for (int q = 0; q < gf.nk; ++q) {
        const int j = (q + 1) / 2;
        const double v = q == 0 ? hf[a] : (q & 1) ? hf[a + j * gf.comp_stride] : hf[a - wsf.off[j] + j * gf.comp_stride];
        if (v == 0.0) continue;
        const int bx = ax + gf.kdx[q], by = ay + gf.kdy[q], bz = az + gf.kdz[q];
        const int px = bx & 1, py = hy ? (by & 1) : 0, pz = hz ? (bz & 1) : 0;
        const bool mid = px | py | pz;
        for (int s = 0; s < (mid ? 2 : 1); ++s) {
          const int sg = s == 0 ? -1 : 1;
          const int jx = (bx + sg * px) / 2, jy = (by + sg * py) / 2, jz = (bz + sg * pz) / 2;
          if (bc_node(gc, bc, jx, jy, jz, &bcv)) continue;
          const int k = wsc.kidx[(jx - ix + 1) + 3 * (jy - iy + 1) + 9 * (jz - lz + 1)];
          if (k < 0) { atomicAdd(bad, 1); continue; }
          acc[k] += wm * v * (mid ? 0.5 : 1.0);
        }
      }
    }
    hc[ic] = acc[0];
    for (int j = 1; j < wsc.nh; ++j) hc[ic + j * gc.comp_stride] = acc[2 * j - 1];
  }
}

// max over free rows of sum_j |a_ij| / a_ii  (positive doubles order like their bit patterns: integer atomicMax)
__global__ void __launch_bounds__(256)
k_wlmax(const __grid_constant__ Grid g, const __grid_constant__ WStencil ws, const double* __restrict__ h,
        unsigned long long* out) {
  const long long total = (long long)g.nn[0] * g.nn[1] * g.nzl;
  double mx = 0.0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long row = t / g.nn[0];
    const int ix = (int)(t - row * g.nn[0]);
    const long long i = (long long)g.PX * (row % g.nn[1]) + g.plane * (row / g.nn[1]) + ix;
    const double d = h[i];
    if (!(d > 0.0)) continue;
    double s = d;
    for (int j = 1; j < ws.nh; ++j) s += fabs(h[i + j * g.comp_stride]) + fabs(h[i - ws.off[j] + j * g.comp_stride]);
    mx = fmax(mx, s / d);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && mx > 0.0) atomicMax(out, (unsigned long long)__double_as_longlong(mx));
}

static int make_wstencil(const Grid& g, WStencil* ws) {
  std::memset(ws, 0, sizeof(*ws));
  ws->nh = 1 + (g.nk - 1) / 2;
  for (int k = 0; k < 27; ++k) ws->kidx[k] = -1;
  for (int k = 0; k < g.nk; ++k) ws->kidx[(g.kdx[k] + 1) + 3 * (g.kdy[k] + 1) + 9 * (g.kdz[k] + 1)] = k;
  for (int j = 1; j < ws->nh; ++j) {
    const int kp = 2 * j - 1, kn = 2 * j;
    if (g.kdx[kn] != -g.kdx[kp] || g.kdy[kn] != -g.kdy[kp] || g.kdz[kn] != -g.kdz[kp] ||
        g.kdx[kp] < 0 || g.kdy[kp] < 0 || g.kdz[kp] < 0)
      PDE_FAIL("stencil offsets are not ordered in (+k, -k) pairs");
    ws->off[j] = g.koff[kp];
    ws->dx[j] = g.kdx[kp]; ws->dy[j] = g.kdy[kp]; ws->dz[j] = g.kdz[kp];
  }
  return 0;
}

// One wave of resident blocks: the grid-stride loop gives every block the same share, so a grid larger than what fits
// at once leaves a second, partly empty wave (the 40-register modes fit 6 blocks of 256 per SM, not 8).
template <int NH, int M>
static int wsweep_blocks(pde_ctx* c, long long total) {
  static int occ = 0;
  if (occ == 0 && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_wsweep<NH, M>, 256, 0) != cudaSuccess) occ = 1;
  const long long want = (total + 255) / 256, cap = (long long)c->sm_count * (occ > 0 ? occ : 1);
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

static int wsweep(pde_ctx* c, const WLevel& L, const BcDev& bc, int mode, const double* x, const double* b,
                  const double* xprev, double* y, double c1, double c2, int slot) {
  const Grid& g = L.g;
  const long long total = (long long)g.nn[0] * g.nn[1] * g.nzl;
  if (total >= (1LL << 32)) PDE_FAIL("weighted multigrid: too many nodes per level");
  double* out = slot >= 0 ? c->scal + slot : nullptr;
#define WSW(NH, M) k_wsweep<NH, M><<<wsweep_blocks<NH, M>(c, total), 256, 0, c->stream>>>( \
                       g, bc, L.ws, L.h.p, x, b, xprev, y, c1, c2, slot >= 0, c->red, out)
#define WSW_NH(NH)                         \
  switch (mode) {                          \
    case W_FIRST: WSW(NH, W_FIRST); break; \
    case W_APPLY: WSW(NH, W_APPLY); break; \
    case W_RESID: WSW(NH, W_RESID); break; \
    default: WSW(NH, W_CHEBY); break;      \
  }
  if (L.ws.nh == 8) { WSW_NH(8) } else if (L.ws.nh == 4) { WSW_NH(4) } else { WSW_NH(2) }
#undef WSW_NH
#undef WSW
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// lmax of D^-1 A: Gershgorin bound from k_wlmax
static int level_lmax(pde_ctx* c, WLevel& L) {
  const long long total = (long long)L.g.nn[0] * L.g.nn[1] * L.g.nzl;
  CUDA_OK(cudaMemsetAsync(c->scal + S_TMP0, 0, sizeof(double), c->stream));
  k_wlmax<<<flat_blocks(c, total, 256), 256, 0, c->stream>>>(L.g, L.ws, L.h.p,
                                                             reinterpret_cast<unsigned long long*>(c->scal + S_TMP0));
  c->launches++;
  CUDA_OK(cudaGetLastError());
  PDE_OK(read_scal(c, S_TMP0, 1, &L.lmax));
  if (!(L.lmax > 0.0)) PDE_FAIL("weighted multigrid: level without a free row");
  return 0;
}

// host copy of a level's half coefficients, indexed like the device field
static int level_to_host(pde_ctx* c, const WLevel& L, std::vector<double>* hh, size_t* base) {
  hh->resize(L.h.bytes / sizeof(double));
  CUDA_OK(cudaMemcpyAsync(hh->data(), L.h.raw, L.h.bytes, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(cudaStreamSynchronize(c->stream));
  *base = (size_t)(L.h.p - L.h.raw);
  return 0;
}

static int build_dense(pde_ctx* c, WLevel& L, const BcDev& bc) {
  const Grid& g = L.g;
  std::vector<long long> idx;
  std::vector<int> dofid;
  const long long n = count_free_and_index(g, bc, 1, &idx, &dofid);
  std::vector<double> hh;
  size_t base;
  PDE_OK(level_to_host(c, L, &hh, &base));
  std::vector<double> A((size_t)n * n, 0.0);
  for (int iz = 0; iz < g.nzl; ++iz)
    for (int iy = 0; iy < g.nn[1]; ++iy)
      for (int ix = 0; ix < g.nn[0]; ++ix) {
        const int di = dofid[((size_t)iz * g.nn[1] + iy) * g.nn[0] + ix];
        if (di < 0) continue;
        const size_t i = base + (size_t)g.PX * iy + (size_t)g.plane * iz + ix;
        A[(size_t)di * n + di] = hh[i];
        for (int j = 1; j < L.ws.nh; ++j) {
          const int jx = ix + L.ws.dx[j], jy = iy + L.ws.dy[j], jz = iz + L.ws.dz[j];
          if (jx >= g.nn[0] || jy >= g.nn[1] || jz >= g.nzl) continue;
          const int dj = dofid[((size_t)jz * g.nn[1] + jy) * g.nn[0] + jx];
          if (dj < 0) continue;
          const double v = hh[i + j * g.comp_stride];
          A[(size_t)di * n + dj] += v;
          A[(size_t)dj * n + di] += v;
        }
      }
  if (dense_inverse_spd(A, (int)n)) PDE_FAIL("weighted multigrid: coarse operator is not positive definite");
  L.n_dense = (int)n;
  CUDA_OK(cudaMalloc(&L.Ainv, A.size() * sizeof(double)));
  CUDA_OK(cudaMalloc(&L.idx, idx.size() * sizeof(long long)));
  CUDA_OK(cudaMemcpyAsync(L.Ainv, A.data(), A.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(cudaMemcpyAsync(L.idx, idx.data(), idx.size() * sizeof(long long), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

int WHierarchy::build(pde_ctx* c, const Grid& g0, const BcDev& bc0, const double* coefA) {
  release();
  bc = bc0;
  const int dim = g0.dim;
  int ax[3], nax;
  internal_axes(dim, ax, &nax);
  int32_t n[3] = {0, 0, 0};
  double Lu[3] = {1, 1, 1};
  for (int q = 0; q < nax; ++q) {
    n[q] = g0.nc[ax[q]];
    Lu[q] = g0.h[ax[q]] * g0.nc[ax[q]];
  }
  int* bad = nullptr;
  CUDA_OK(cudaMalloc(&bad, sizeof(int)));
  struct BadRel { int* p; ~BadRel() { cudaFree(p); } } badrel{bad};
  CUDA_OK(cudaMemsetAsync(bad, 0, sizeof(int), c->stream));
  for (int level = 0;; ++level) {
    std::unique_ptr<WLevel> L(new WLevel());
    if (level == 0) L->g = g0;
    else PDE_OK(make_grid(dim, n, Lu, 0, 1, &L->g));
    const Grid& g = L->g;
    PDE_OK(make_wstencil(g, &L->ws));
    PDE_OK(L->h.alloc(c, g, L->ws.nh));
    PDE_OK(L->xa.alloc(c, g, 1));
    PDE_OK(L->xb.alloc(c, g, 1));
    PDE_OK(L->r.alloc(c, g, 1));
    if (level > 0) PDE_OK(L->b.alloc(c, g, 1));
    const long long total = (long long)g.nn[0] * g.nn[1] * g.nzl;
    if (level == 0) {
      k_wpack<<<flat_blocks(c, total, 256), 256, 0, c->stream>>>(g, bc, L->ws, coefA, L->h.p);
    } else {
      const WLevel& F = *lv.back();
      k_wgalerkin<<<flat_blocks(c, total, 128), 128, 0, c->stream>>>(F.g, g, bc, F.ws, L->ws, F.h.p, L->h.p, bad);
    }
    c->launches++;
    CUDA_OK(cudaGetLastError());
    PDE_OK(level_lmax(c, *L));
    lv.push_back(std::move(L));
    // coarsen while every axis halves evenly and the coarse grid keeps a free node
    bool can = true;
    int32_t nc2[3] = {0, 0, 0};
    for (int q = 0; q < nax; ++q) {
      if (n[q] % 2 != 0 || n[q] < 2) can = false;
      nc2[q] = n[q] / 2;
    }
    if (can) {
      Grid gc;
      PDE_OK(make_grid(dim, nc2, Lu, 0, 1, &gc));
      if ((long long)gc.nn[0] * gc.nn[1] * gc.nzl <= 200000 && count_free_and_index(gc, bc, 1, nullptr, nullptr) <= 0)
        can = false;
    }
    if (!can) break;
    for (int q = 0; q < nax; ++q) n[q] = nc2[q];
  }
  int nbad = 0;
  CUDA_OK(cudaMemcpyAsync(&nbad, bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(cudaStreamSynchronize(c->stream));
  if (nbad) PDE_FAIL("weighted multigrid: Galerkin product left the Kuhn stencil (" + std::to_string(nbad) + " entries)");
  WLevel& Lc = *lv.back();
  if (lv.size() > 1 && (long long)Lc.g.nn[0] * Lc.g.nn[1] * Lc.g.nzl <= 4 * PDE_DENSE_MAX) {
    const long long nfree = count_free_and_index(Lc.g, bc, 1, nullptr, nullptr);
    if (nfree > 0 && nfree <= PDE_DENSE_MAX) PDE_OK(build_dense(c, Lc, bc));
  }
  return 0;
}

void WHierarchy::release() {
  for (auto& L : lv) {
    L->h.release(); L->b.release(); L->xa.release(); L->xb.release(); L->r.release();
    if (L->Ainv) cudaFree(L->Ainv);
    if (L->idx) cudaFree(L->idx);
  }
  lv.clear();
}

// Chebyshev(Jacobi) on [lmax/ratio, lmax], the recurrence of solver.cu's first-kind smoother.  x lives in *cur on
// entry and exit.  dot_slot >= 0: the last sweep also leaves sum b.x_new there (it must be a general sweep).
static int wsmooth(pde_ctx* c, const WHierarchy& H, WLevel& L, const double* b, double** cur, double** oth,
                   int sweeps, bool zero_guess, double ratio, int dot_slot) {
  const double lmin = L.lmax / ratio;
  const double theta = 0.5 * (L.lmax + lmin), delta = 0.5 * (L.lmax - lmin), sigma = theta / delta;
  double rho = 1.0 / sigma;
  int k0 = 0;
  if (zero_guess) {
    PDE_OK(wsweep(c, L, H.bc, W_FIRST, nullptr, b, nullptr, *cur, 0.0, 1.0 / theta, -1));
    k0 = 1;
  }
  for (int k = k0; k < sweeps; ++k) {
    double c1 = 0.0, c2 = 1.0 / theta;
    if (k > 0) {
      const double rn = 1.0 / (2.0 * sigma - rho);
      c1 = rn * rho;
      c2 = 2.0 * rn / delta;
      rho = rn;
    }
    // x_{k-1}: none on a restart, zero after the first sweep from a zero guess, else the other buffer
    const double* xprev = (k == 0 || (zero_guess && k == 1)) ? nullptr : *oth;
    PDE_OK(wsweep(c, L, H.bc, W_CHEBY, *cur, b, xprev, *oth, c1, c2, k == sweeps - 1 ? dot_slot : -1));
    std::swap(*cur, *oth);
  }
  return 0;
}

// z = V(b0); the last level-0 post-sweep leaves sum b0.z in dot_slot
int wvcycle(pde_ctx* c, WHierarchy& H, const double* b0, double** z_out, int dot_slot) {
  const int nl = H.levels();
  std::vector<double*> cur(nl), oth(nl);
  for (int l = 0; l < nl; ++l) { cur[l] = H.lv[l]->xa.p; oth[l] = H.lv[l]->xb.p; }
  for (int l = 0; l + 1 < nl; ++l) {
    WLevel& L = *H.lv[l];
    const double* b = l == 0 ? b0 : L.b.p;
    PDE_OK(wsmooth(c, H, L, b, &cur[l], &oth[l], H.nu, true, H.ratio, -1));
    PDE_OK(wsweep(c, L, H.bc, W_RESID, cur[l], b, nullptr, L.r.p, 0.0, 0.0, -1));
    PDE_OK(launch_restrict(c, L.g, H.lv[l + 1]->g, H.bc, 1, L.r.p, H.lv[l + 1]->b.p));
  }
  WLevel& Lc = *H.lv[nl - 1];
  if (Lc.n_dense > 0) PDE_OK(launch_dense_solve(c, Lc.n_dense, Lc.Ainv, Lc.idx, Lc.b.p, cur[nl - 1]));
  else PDE_OK(wsmooth(c, H, Lc, Lc.b.p, &cur[nl - 1], &oth[nl - 1], H.coarse_sweeps, true, 30.0, -1));
  for (int l = nl - 2; l >= 0; --l) {
    WLevel& L = *H.lv[l];
    PDE_OK(launch_prolong_add(c, L.g, H.lv[l + 1]->g, H.bc, 1, cur[l + 1], cur[l]));
    PDE_OK(wsmooth(c, H, L, l == 0 ? b0 : L.b.p, &cur[l], &oth[l], H.nu, false, H.ratio, l == 0 ? dot_slot : -1));
  }
  *z_out = cur[0];
  return 0;
}

// The recurrence of pcg_solve (GMG branch): device scalars, the x update deferred into the p update, a poll per
// iteration.  The flat vector kernels only use ncomp from the operator description.
int wmg_pcg(pde_ctx* c, WHierarchy& h, double* x, double* r, double* p, double* q, double bnorm2,
            const pde_solver_opts& o, pde_stats* st) {
  if (h.levels() < 2) PDE_FAIL("weighted multigrid needs at least two levels");
  WLevel& L0 = *h.lv[0];
  const Grid& g = L0.g;
  OpDev one;
  one.ncomp = 1;
  st->solves += 1;
  st->levels = h.levels();
  if (!(bnorm2 > 0.0)) { st->final_relres = 0.0; return 0; }
  const double tol2 = o.rtol * o.rtol * bnorm2;
  double* z = nullptr;
  PDE_OK(wvcycle(c, h, r, &z, S_RHO0));
  PDE_OK(launch_dot(c, g, 1, r, r, S_RHO0 + 1));
  PDE_OK(launch_cg_pupdate(c, g, one, p, z, S_RHO0, S_RHO0, 1, 0));
  double rr;
  PDE_OK(read_scal(c, S_RHO0 + 1, 1, &rr));
  int it = 0;
  bool conv = rr <= tol2;
  while (!conv && it < o.max_iters) {
    const int sr = 2 * (it & 1), sn = 2 * (1 - (it & 1));
    PDE_OK(wsweep(c, L0, h.bc, W_APPLY, p, nullptr, nullptr, q, 0.0, 0.0, S_XY));     // q = A p, p.q
    PDE_OK(launch_cg_update(c, g, one, nullptr, r, p, q, sr, S_XY, sn, sn + 1, 0));  // r -= a q, r.r
    PDE_OK(wvcycle(c, h, r, &z, sn));                                                // z = V(r), r.z
    PDE_OK(launch_cg_pupdate(c, g, one, p, z, sr, sn, 0, 0, x, S_XY));               // x += a p, p = z + b p
    ++it;
    PDE_OK(read_scal(c, sn + 1, 1, &rr));
    if (!(rr == rr)) PDE_FAIL("weighted GMG-PCG broke down (NaN residual)");
    conv = rr <= tol2;
  }
  st->iters_total += it;
  st->final_relres = std::sqrt(rr / bnorm2);
  if (!conv) st->converged = 0;
  return 0;
}

int wmg_level_coefs(pde_ctx* c, const WHierarchy& h, int level, double* out) {
  if (level < 0 || level >= h.levels()) PDE_FAIL("no such multigrid level");
  const WLevel& L = *h.lv[level];
  const Grid& g = L.g;
  std::vector<double> hh;
  size_t base;
  PDE_OK(level_to_host(c, L, &hh, &base));
  const size_t nv = (size_t)g.nn[0] * g.nn[1] * g.nzl;
  for (int k = 0; k < g.nk; ++k) {
    const int j = (k + 1) / 2;
    for (int iz = 0; iz < g.nzl; ++iz)
      for (int iy = 0; iy < g.nn[1]; ++iy)
        for (int ix = 0; ix < g.nn[0]; ++ix) {
          const size_t i = base + (size_t)g.PX * iy + (size_t)g.plane * iz + ix;
          double v;
          if (k == 0) v = hh[i];
          else if (k & 1) v = hh[i + j * g.comp_stride];
          else v = hh[i - L.ws.off[j] + j * g.comp_stride];
          out[(size_t)k * nv + ((size_t)iz * g.nn[1] + iy) * g.nn[0] + ix] = v;
        }
  }
  return 0;
}
