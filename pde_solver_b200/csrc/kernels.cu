// Generic (table-driven) sm_100a kernels: correct for every node class, dimension and BC set.
// The specialised streaming kernels for the 3D hot paths live in stencil3d.cu.
//
// Replaces, matrix-free, what the reference does through DOLFIN assembly + PETSc LU:
//   k_stencil        : y = bs*B + as*(A x)  /  Chebyshev sweep   (forms fenics_mcp_server.py:261-262,
//                      304-305, 393-394, 433-434, 657-658, 702-703, 1527-1528, 1677-1678, 1827-1828)
//   k_cg_*           : the linear solve of solve(a == L, u, bcs)  (:311, 440, 709, 1538, 1688, 1838)
//   k_cell_rhs       : von-Mises / axial stress-strain load of project(eq_expr, Vs) (:1541-1546,
//                      1691-1714, 1841-1862)
//   k_mesh_*         : IntervalMesh/RectangleMesh/BoxMesh + P1 dof maps (:229-230, 369-370, 533-535)
#include <cstring>

#include "device.cuh"
#include "tma.cuh"

// ----------------------------------------------------------------------------------------------
// generic stencil kernel
// ----------------------------------------------------------------------------------------------
template <int NC>
struct IntCoef {
  double c[PDE_NOFF][NC * NC];
};

struct StencilDev {
  const double* x;
  const double* b;
  double* y;
  const double* xprev;
  int prev_mode;
  double bconst[3];
  double bscale, ascale, c1, c2, s0;
  int do_reduce;
  int first2;
  double* defer;   // face rows: leave the block sums here instead of finalizing
};

template <int NC, bool CHEBY>
__global__ void __launch_bounds__(128)
k_stencil(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc,
          const __grid_constant__ IntCoef<NC> ic, const double* __restrict__ coef,
          const double* __restrict__ dinv, const double* __restrict__ load,
          const __grid_constant__ StencilDev a, ReduceBuf red, double* red_out) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  double acc_xy = 0.0, acc_yy = 0.0;
  const bool fast3d = (g.nk == PDE_NOFF);
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const int gz = lz + g.z0;
    const long long rbase = (long long)g.PX * iy + g.plane * lz;
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const long long idx = rbase + ix;
      double bcv;
      const bool isdir = bc_node(g, bc, ix, iy, gz, &bcv);
      if (isdir) {
#pragma unroll
        for (int i = 0; i < NC; ++i) {
          if (CHEBY) {
            a.y[idx + i * g.comp_stride] = a.x[idx + i * g.comp_stride];
          } else if (a.y) {
            a.y[idx + i * g.comp_stride] = 0.0;
          }
        }
        continue;
      }
      const int cls = node_class(g, ix, iy, gz);
      double acc[NC];
#pragma unroll
      for (int i = 0; i < NC; ++i) acc[i] = 0.0;
      if (fast3d && cls == 13) {
#pragma unroll
        for (int k = 0; k < PDE_NOFF; ++k) {
          const long long off = kOffDdev(k, g.PX, g.plane);
          double xv[NC];
#pragma unroll
          for (int j = 0; j < NC; ++j) xv[j] = a.x[idx + off + j * g.comp_stride];
#pragma unroll
          for (int i = 0; i < NC; ++i)
#pragma unroll
            for (int j = 0; j < NC; ++j) acc[i] = fma(ic.c[k][i * NC + j], xv[j], acc[i]);
        }
      } else if (g.nk == 7 && cls == 13) {
        // 2-D interior rows (internal axes x, z): the seven Kuhn offsets with constant-bank coefficients
        constexpr int K2[7] = {0, 1, 2, 5, 6, 9, 10};
#pragma unroll
        for (int q = 0; q < 7; ++q) {
          const int k = K2[q];
          const long long off = kOffDdev(k, g.PX, g.plane);
          double xv[NC];
#pragma unroll
          for (int j = 0; j < NC; ++j) xv[j] = a.x[idx + off + j * g.comp_stride];
#pragma unroll
          for (int i = 0; i < NC; ++i)
#pragma unroll
            for (int j = 0; j < NC; ++j) acc[i] = fma(ic.c[k][i * NC + j], xv[j], acc[i]);
        }
      } else {
        for (int k = 0; k < g.nk; ++k) {
          const double* cf = coef + ((size_t)cls * PDE_NOFF + g.kidx[k]) * (NC * NC);
          const long long off = g.koff[k];
          double xv[NC];
#pragma unroll
          for (int j = 0; j < NC; ++j) xv[j] = a.x[idx + off + j * g.comp_stride];
#pragma unroll
          for (int i = 0; i < NC; ++i)
#pragma unroll
            for (int j = 0; j < NC; ++j) acc[i] = fma(__ldg(cf + i * NC + j), xv[j], acc[i]);
        }
      }
      const double ld = a.b ? 0.0 : __ldg(load + cls);
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const long long ii = idx + i * g.comp_stride;
        const double B = a.b ? a.b[ii] : a.bconst[i] * ld;
        if (CHEBY) {
          const double di = __ldg(dinv + cls * NC + i);
          double dn, yv, Bv;
          if (a.first2) {  // x holds the right-hand side; x1 = d1 = s0 D^-1 b (uniform diagonal)
            Bv = a.x[ii];
            const double d1 = a.s0 * di * Bv;
            dn = a.c1 * d1 + a.c2 * di * (Bv - a.s0 * di * acc[i]);
            yv = d1 + dn;
          } else {
            Bv = B;
            const double xo = a.x[ii];
            const double dprev = a.prev_mode == 1 ? xo - a.xprev[ii]
                               : (a.prev_mode == 2 ? xo : (a.prev_mode == 3 ? xo - a.s0 * di * B : 0.0));
            dn = a.c1 * dprev + a.c2 * di * (B - acc[i]);
            yv = xo + dn;
          }
          a.y[ii] = yv;
          if (a.do_reduce) acc_xy = fma(Bv, yv, acc_xy);
        } else {
          const double yv = a.bscale * B + a.ascale * acc[i];
          if (a.y) a.y[ii] = yv;
          if (a.do_reduce) {
            acc_xy = fma(a.x[ii], yv, acc_xy);
            acc_yy = fma(yv, yv, acc_yy);
          }
        }
      }
    }
  }
  if (a.do_reduce) {
    if (CHEBY) {
      double v[1] = {acc_xy};
      block_reduce_finalize<1>(v, red, red_out);
    } else {
      double v[2] = {acc_xy, acc_yy};
      block_reduce_finalize<2>(v, red, red_out);
    }
  }
}

template <int NC>
static int launch_stencil_t(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a) {
  IntCoef<NC> ic;
  for (int k = 0; k < PDE_NOFF; ++k)
    for (int q = 0; q < NC * NC; ++q) ic.c[k][q] = op.h_int[k * NC * NC + q];
  StencilDev sd;
  sd.x = a.x; sd.b = a.b; sd.y = a.y; sd.xprev = a.xprev; sd.prev_mode = a.prev_mode;
  for (int i = 0; i < 3; ++i) sd.bconst[i] = a.bconst[i];
  sd.bscale = a.bscale; sd.ascale = a.ascale; sd.c1 = a.c1; sd.c2 = a.c2; sd.s0 = a.s0;
  sd.first2 = a.cheby == 2;
  sd.defer = nullptr;
  sd.do_reduce = a.reduce_slot_xy >= 0;
  RowLaunch rl = row_launch(c, g);
  double* out = sd.do_reduce ? c->scal + a.reduce_slot_xy : nullptr;
  if (a.cheby)
    k_stencil<NC, true><<<rl.grid, rl.block, 0, c->stream>>>(g, bc, ic, op.coef, op.dinv, op.load, sd, c->red, out);
  else
    k_stencil<NC, false><<<rl.grid, rl.block, 0, c->stream>>>(g, bc, ic, op.coef, op.dinv, op.load, sd, c->red, out);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int launch_stencil_generic(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a) {
  switch (op.ncomp) {
    case 1: return launch_stencil_t<1>(c, g, bc, op, a);
    case 2: return launch_stencil_t<2>(c, g, bc, op, a);
    case 3: return launch_stencil_t<3>(c, g, bc, op, a);
  }
  PDE_FAIL("unsupported component count");
}

// ----------------------------------------------------------------------------------------------
// PCG vector kernels (row-structured: the Jacobi diagonal depends on the node class)
// ----------------------------------------------------------------------------------------------
template <int NC>
__global__ void __launch_bounds__(128)
k_cg_update(const __grid_constant__ Grid g, const double* __restrict__ dinv, double* __restrict__ x,
            double* __restrict__ r, const double* __restrict__ p, const double* __restrict__ q,
            const double* __restrict__ scal, int s_rho, int s_pap, ReduceBuf red, double* out_rho_new,
            double* out_rr) {
  const double pap = scal[s_pap], rho = scal[s_rho];
  const double alpha = pap > 0.0 ? rho / pap : 0.0;
  const long long rows = (long long)g.nn[1] * g.nzl;
  double rz = 0.0, rr = 0.0;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const long long rbase = (long long)g.PX * iy + g.plane * lz;
    const int cyz = 3 * axis_class(iy, g.nn[1]) + 9 * axis_class(lz + g.z0, g.nzg);
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const int cls = axis_class(ix, g.nn[0]) + cyz;
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const long long ii = rbase + ix + i * g.comp_stride;
        const double pv = p[ii], qv = q[ii];
        x[ii] = fma(alpha, pv, x[ii]);
        const double rv = fma(-alpha, qv, r[ii]);
        r[ii] = rv;
        rr = fma(rv, rv, rr);
        rz = fma(rv * __ldg(dinv + cls * NC + i), rv, rz);
      }
    }
  }
  double v[2] = {rz, rr};
  // the caller guarantees out_rr == out_rho_new + 1: one finalize writes both sums
  block_reduce_finalize<2>(v, red, out_rho_new);
  (void)out_rr;
}

template <int NC>
__global__ void __launch_bounds__(128)
k_cg_pupdate(const __grid_constant__ Grid g, const double* __restrict__ dinv, double* __restrict__ p,
             const double* __restrict__ rz, const double* __restrict__ scal, int s_rho, int s_rho_new,
             int first, int jacobi) {
  double beta = 0.0;
  if (!first) {
    const double rho = scal[s_rho];
    beta = rho > 0.0 ? scal[s_rho_new] / rho : 0.0;
  }
  const long long rows = (long long)g.nn[1] * g.nzl;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const long long rbase = (long long)g.PX * iy + g.plane * lz;
    const int cyz = 3 * axis_class(iy, g.nn[1]) + 9 * axis_class(lz + g.z0, g.nzg);
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const int cls = axis_class(ix, g.nn[0]) + cyz;
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const long long ii = rbase + ix + i * g.comp_stride;
        const double z = jacobi ? rz[ii] * __ldg(dinv + cls * NC + i) : rz[ii];
        p[ii] = first ? z : fma(beta, p[ii], z);
      }
    }
  }
}

#define DISPATCH_NC(nc, CALL)                       \
  switch (nc) {                                     \
    case 1: { constexpr int NC = 1; CALL; } break;  \
    case 2: { constexpr int NC = 2; CALL; } break;  \
    case 3: { constexpr int NC = 3; CALL; } break;  \
    default: PDE_FAIL("unsupported component count"); \
  }

// ----------------------------------------------------------------------------------------------
// face rows: the non-Dirichlet nodes on the faces of the box have incomplete element patches, so their
// stencil coefficients come from the 27-class table.  The streaming kernel (stencil3d.cu) skips them;
// this kernel computes them right after it, one thread per face node (edges / corners counted once).
// ----------------------------------------------------------------------------------------------
struct FaceSet {
  int nface;
  int axis[12], fixed[12];        // fixed axis and its index (z: LOCAL plane); up to two layers per face
  int lo[12][2], cnt[12][2];      // the two varying axes (ascending axis order): start and count
  int tiles0[12];                 // tiles of FACE_TU nodes along the first varying axis
  int tstart[13];                 // prefix sums of the tile counts: one CTA per FACE_TU x FACE_TV tile
};
#define FACE_TU 32
#define FACE_TV 8
#define FACE_NT (FACE_TU * FACE_TV)

// One CTA per 32 x 8 tile of a face (warp = 32 consecutive nodes along the first varying axis, the 8 warps are 8
// consecutive lines along the second): the three lines / planes a node needs are shared with the warps next to it, so
// most of the 15 x NC loads hit L1.  FULL: the 3-D stencil with all 15 offsets in table order.  The kernel is latency
// bound (a few wide dependent steps, little data), so everything a node reads from HBM - its 15 x NC neighbours, its
// own x / b / x_prev - is requested FIRST; while those loads fly the block marks the node classes it meets and copies
// those rows of the class table into shared memory (a face tile meets one to three of the 27), and the products then
// read the coefficients as warp-uniform shared-memory broadcasts.
// History on the cantilever faces of 1280x256x256 (1.38 M nodes): 141 us with per-node __ldg'ed coefficients and a
// rolled offset loop, against 0.75 ms for the whole interior sweep.
#ifndef FACE_MINB
#define FACE_MINB 2
#endif
template <int NC, bool CHEBY, bool FULL>
__global__ void __launch_bounds__(FACE_NT, FULL ? FACE_MINB : 1)
k_face_rows(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc, const __grid_constant__ FaceSet fs,
            const double* __restrict__ coef, const double* __restrict__ dinv, const double* __restrict__ load,
            const __grid_constant__ StencilDev a, ReduceBuf red, double* red_out) {
  constexpr int ROW = PDE_NOFF * NC * NC;
  constexpr int ROWP = (ROW + 1) / 2 * 2;   // rows stay 16-byte aligned
  __shared__ __align__(16) double s_coef[FULL ? PDE_NCLASS * ROWP : 2];
  __shared__ unsigned s_mask, s_nz[PDE_NCLASS];
  __shared__ double s_dinv[PDE_NCLASS * NC];
  double acc_xy = 0.0, acc_yy = 0.0;
  {
    const int tile = blockIdx.x;
    int f = 0;
#pragma unroll
    for (int q = 1; q < 12; ++q) f += (q < fs.nface && tile >= fs.tstart[q]) ? 1 : 0;
    const int tl = tile - fs.tstart[f];
    const int tv = tl / fs.tiles0[f], tu = tl - tv * fs.tiles0[f];
    const int ul = tu * FACE_TU + (threadIdx.x & (FACE_TU - 1)), vl = tv * FACE_TV + (threadIdx.x / FACE_TU);
    bool live = ul < fs.cnt[f][0] && vl < fs.cnt[f][1];
    const int u = fs.lo[f][0] + ul, v = fs.lo[f][1] + vl;
    int ix, iy, lz;
    if (fs.axis[f] == 0) { ix = fs.fixed[f]; iy = u; lz = v; }
    else if (fs.axis[f] == 1) { ix = u; iy = fs.fixed[f]; lz = v; }
    else { ix = u; iy = v; lz = fs.fixed[f]; }
    int cls = 13;
    if (live) {
      double bcv;
      if (bc_node(g, bc, ix, iy, lz + g.z0, &bcv)) live = false;  // Dirichlet rows were written (masked) by the main kernel
      cls = node_class(g, ix, iy, lz + g.z0);
    }
    // 32-bit element offsets from three component bases (the host checks that a component triple fits 2^31 elements):
    // one add + one widening multiply-add per load instead of a 64-bit address rebuild
    const long long idxl = live ? (long long)g.PX * iy + g.plane * lz + ix : 0;   // dead lanes read around node 0 (in bounds)
    const int idx = (int)idxl;   // FULL only
    const double* xc[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) xc[j] = a.x + j * g.comp_stride;
    double xv[PDE_NOFF][NC], xo[NC], bv[NC], pv[NC];
    if (FULL) {
#pragma unroll
      for (int k = 0; k < PDE_NOFF; ++k) {
        const int off = (int)kOffDdev(k, g.PX, g.plane);
#pragma unroll
        for (int j = 0; j < NC; ++j) xv[k][j] = xc[j][idx + off];
      }
    }
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      xo[i] = xc[i][idxl];
      bv[i] = a.b ? (a.b + i * g.comp_stride)[idxl] : 0.0;
      pv[i] = (CHEBY && a.prev_mode == 1) ? (a.xprev + i * g.comp_stride)[idxl] : 0.0;
    }
    if (FULL) {
      if (CHEBY && a.first2)
        for (int e = threadIdx.x; e < PDE_NCLASS * NC; e += blockDim.x) s_dinv[e] = __ldg(dinv + e);
      if (threadIdx.x < PDE_NCLASS) s_nz[threadIdx.x] = 0u;
      if (threadIdx.x == 0) s_mask = 0u;
      __syncthreads();
      const unsigned mine = __reduce_or_sync(0xffffffffu, live ? (1u << cls) : 0u);
      if ((threadIdx.x & 31) == 0 && mine) atomicOr(&s_mask, mine);
      __syncthreads();
      for (unsigned m = s_mask; m; m &= m - 1) {
        const int k = __ffs(m) - 1;
        for (int e = threadIdx.x; e < ROW; e += blockDim.x) {
          const double cv = __ldg(coef + (size_t)k * ROW + e);
          s_coef[k * ROWP + e] = cv;
          if (cv != 0.0) atomicOr(&s_nz[k], 1u << (e / (NC * NC)));   // offsets whose block is not identically zero
        }
      }
      __syncthreads();
    }
    if (live) {
      double acc[NC];
#pragma unroll
      for (int i = 0; i < NC; ++i) acc[i] = 0.0;
      if (FULL && CHEBY && a.first2) {
        // fused first two sweeps: the loaded field is the right-hand side b; x1 = s0 D^-1 b with the class diagonal of
        // EVERY neighbour (that is why the layer next to a natural face is computed here too)
#pragma unroll
        for (int k = 0; k < PDE_NOFF; ++k) {
          const int jx = ix + kOffDcomp(k, 0), jy = iy + kOffDcomp(k, 1), jz = lz + g.z0 + kOffDcomp(k, 2);
          const bool in = jx >= 0 && jx < g.nn[0] && jy >= 0 && jy < g.nn[1] && jz >= 0 && jz < g.nzg;
          const int ck = in ? node_class(g, jx, jy, jz) : 13;
#pragma unroll
          for (int j = 0; j < NC; ++j) xv[k][j] *= a.s0 * s_dinv[ck * NC + j];
        }
      }
      if (FULL) {
        const double* cf = s_coef + cls * ROWP;
        const unsigned nz = s_nz[cls];
        // a face node has no neighbours beyond the face: a third of its blocks are zero (warp-uniform skip)
#pragma unroll
        for (int k = 0; k < PDE_NOFF; ++k) {
          if (!((nz >> k) & 1u)) continue;
#pragma unroll
          for (int i = 0; i < NC; ++i)
#pragma unroll
            for (int j = 0; j < NC; ++j) acc[i] = fma(cf[k * NC * NC + i * NC + j], xv[k][j], acc[i]);
        }
      } else {
        for (int k = 0; k < g.nk; ++k) {
          const double* cf = coef + ((size_t)cls * PDE_NOFF + g.kidx[k]) * (NC * NC);
          const long long off = g.koff[k];
          double xk[NC];
#pragma unroll
          for (int j = 0; j < NC; ++j) xk[j] = a.x[idxl + off + j * g.comp_stride];
#pragma unroll
          for (int i = 0; i < NC; ++i)
#pragma unroll
            for (int j = 0; j < NC; ++j) acc[i] = fma(__ldg(cf + i * NC + j), xk[j], acc[i]);
        }
      }
      const double ld = a.b ? 0.0 : __ldg(load + cls);
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const double B = a.b ? bv[i] : a.bconst[i] * ld;
        if (CHEBY && a.first2) {
          // xo = b (raw), xv[0] = x1 of this node: y = (1 + c1) x1 + c2 D^-1 (b - A x1)
          const double yv = fma(1.0 + a.c1, xv[0][i], a.c2 * s_dinv[cls * NC + i] * (xo[i] - acc[i]));
          (a.y + i * g.comp_stride)[idxl] = yv;
        } else if (CHEBY) {
          const double di = __ldg(dinv + cls * NC + i);
          const double dprev = a.prev_mode == 1 ? xo[i] - pv[i]
                             : (a.prev_mode == 2 ? xo[i] : (a.prev_mode == 3 ? xo[i] - a.s0 * di * B : 0.0));
          const double dn = a.c1 * dprev + a.c2 * di * (B - acc[i]);
          const double yv = xo[i] + dn;
          (a.y + i * g.comp_stride)[idxl] = yv;
          acc_xy = fma(B, yv, acc_xy);
        } else {
          const double yv = a.bscale * B + a.ascale * acc[i];
          if (a.y) (a.y + i * g.comp_stride)[idxl] = yv;
          acc_xy = fma(xo[i], yv, acc_xy);
          acc_yy = fma(yv, yv, acc_yy);
        }
      }
    }
  }
  if (a.do_reduce && a.defer) {
    // deferred: plain block sums, picked up by the finalize of the sweep kernel that follows
    __shared__ double sm2[2][FACE_NT / 32];
    double v[2] = {acc_xy, acc_yy};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v[i] += __shfl_down_sync(0xffffffffu, v[i], o);
      if ((threadIdx.x & 31) == 0) sm2[i][threadIdx.x >> 5] = v[i];
    }
    __syncthreads();
    if (threadIdx.x < 2) {
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < FACE_NT / 32; ++w) t += sm2[threadIdx.x][w];
      a.defer[(size_t)blockIdx.x * RED_MAX_VALS + threadIdx.x] = t;
    }
  } else if (a.do_reduce) {
    if (CHEBY) {
      double v[1] = {acc_xy};
      block_reduce_finalize<1, true>(v, red, red_out);
    } else {
      double v[2] = {acc_xy, acc_yy};
      block_reduce_finalize<2, true>(v, red, red_out);
    }
  }
}

// ---- k_face_tile: the 3-D three-component face rows with the neighbourhood staged by ONE TMA load per CTA ------------
// k_face_rows keeps the 45 neighbour values of a node in registers (128 registers, 16 warps/SM) and is bound by the
// latency of its scattered loads.  Here the CTA of a 32 x 8 face tile fetches the whole neighbourhood box - the tile grown
// by one node in its two face directions, three layers across the face, all components - with a single
// cp.async.bulk.tensor (out-of-domain parts arrive as zeros, ghost planes hold the halo), the class-table rows are staged
// while it flies, and every node then works out of shared memory: a third of the registers, one bulk request instead
// of 11 520 scattered ones per CTA.
//   box extents (x, y, z): x faces (4, 34, 10), y faces (36, 3, 10), z faces (36, 10, 3); the x start is rounded down to an
//   even column (TMA start coordinates must be 16-byte aligned), which the extents 4 / 36 leave room for.
#define FT_BOX 4096   // doubles per component group: max(4*34*10, 36*3*10, 36*10*3) * 3 = 4080
template <bool CHEBY>
__global__ void __launch_bounds__(FACE_NT, 4)
k_face_tile(const __grid_constant__ CUtensorMap tm0, const __grid_constant__ CUtensorMap tm1,
            const __grid_constant__ CUtensorMap tm2, const __grid_constant__ Grid g, const __grid_constant__ BcDev bc,
            const __grid_constant__ FaceSet fs, const double* __restrict__ coef, const double* __restrict__ dinv,
            const double* __restrict__ load, const __grid_constant__ StencilDev a, ReduceBuf red, double* red_out) {
  constexpr int NC = 3;
  constexpr int ROW = PDE_NOFF * NC * NC;
  constexpr int ROWP = (ROW + 1) / 2 * 2;
  extern __shared__ __align__(128) double s_box[];   // FT_BOX doubles (dynamic: static shared memory ends at 48 KB)
  constexpr int NSLOT = 8;   // class-table rows a tile can meet: face, two edges, a corner (and the interior in layer 1)
  __shared__ __align__(16) double s_coef[NSLOT * ROWP];
  __shared__ unsigned s_mask, s_nz[PDE_NCLASS];
  __shared__ double s_dinv[PDE_NCLASS * NC];
  __shared__ __align__(8) uint64_t s_bar;
  double acc_xy = 0.0, acc_yy = 0.0;
  const int tile = blockIdx.x;
  int f = 0;
#pragma unroll
  for (int q = 1; q < 12; ++q) f += (q < fs.nface && tile >= fs.tstart[q]) ? 1 : 0;
  const int tl = tile - fs.tstart[f];
  const int tv = tl / fs.tiles0[f], tu = tl - tv * fs.tiles0[f];
  const int u0 = fs.lo[f][0] + tu * FACE_TU, v0 = fs.lo[f][1] + tv * FACE_TV;   // first node of the tile
  const int axis = fs.axis[f], fixed = fs.fixed[f];
  // box origin (node coordinates) and extents
  int xs, ys, zs, E0, E1, E2;
  if (axis == 0) { xs = (fixed - 1) & ~1; ys = u0 - 1; zs = v0 - 1; E0 = 4; E1 = FACE_TU + 2; E2 = FACE_TV + 2; }
  else if (axis == 1) { xs = (u0 - 1) & ~1; ys = fixed - 1; zs = v0 - 1; E0 = FACE_TU + 4; E1 = 3; E2 = FACE_TV + 2; }
  else { xs = (u0 - 1) & ~1; ys = v0 - 1; zs = fixed - 1; E0 = FACE_TU + 4; E1 = FACE_TV + 2; E2 = 3; }
  const uint32_t bar = smem_u32(&s_bar);
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(bar, (uint32_t)(E0 * E1 * E2 * NC * 8));
    const CUtensorMap* tm = axis == 0 ? &tm0 : (axis == 1 ? &tm1 : &tm2);
    tma_load_4d(smem_u32(s_box), tm, xs, ys, zs + PDE_NG, 0, bar);
    s_mask = 0u;
  }
  const int ul = threadIdx.x & (FACE_TU - 1), vl = threadIdx.x / FACE_TU;
  bool live = tu * FACE_TU + ul < fs.cnt[f][0] && tv * FACE_TV + vl < fs.cnt[f][1];
  const int u = u0 + ul, v = v0 + vl;
  int ix, iy, lz;
  if (axis == 0) { ix = fixed; iy = u; lz = v; }
  else if (axis == 1) { ix = u; iy = fixed; lz = v; }
  else { ix = u; iy = v; lz = fixed; }
  int cls = 13;
  if (live) {
    double bcv;
    if (bc_node(g, bc, ix, iy, lz + g.z0, &bcv)) live = false;  // Dirichlet rows were written (masked) by the main kernel
    cls = node_class(g, ix, iy, lz + g.z0);
  }
  const long long idxl = live ? (long long)g.PX * iy + g.plane * lz + ix : 0;
  // own right-hand side / previous iterate: the only scattered loads left (issued before the staging below)
  double bv[NC], pv[NC];
#pragma unroll
  for (int i = 0; i < NC; ++i) {
    bv[i] = a.b ? (a.b + i * g.comp_stride)[idxl] : 0.0;
    pv[i] = (CHEBY && a.prev_mode == 1) ? (a.xprev + i * g.comp_stride)[idxl] : 0.0;
  }
  if (CHEBY && a.first2)
    for (int e = threadIdx.x; e < PDE_NCLASS * NC; e += blockDim.x) s_dinv[e] = __ldg(dinv + e);
  if (threadIdx.x < PDE_NCLASS) s_nz[threadIdx.x] = 0u;
  __syncthreads();
  const unsigned mine = __reduce_or_sync(0xffffffffu, live ? (1u << cls) : 0u);
  if ((threadIdx.x & 31) == 0 && mine) atomicOr(&s_mask, mine);
  __syncthreads();
  const unsigned cmask = s_mask;
  const bool slots_ok = __popc(cmask) <= NSLOT;       // always, by the geometry of a 2-D tile; otherwise read the table
  if (slots_ok) {
    int slot = 0;
    for (unsigned m = cmask; m; m &= m - 1, ++slot) {
      const int k = __ffs(m) - 1;
      for (int e = threadIdx.x; e < ROW; e += blockDim.x) {
        const double cv = __ldg(coef + (size_t)k * ROW + e);
        s_coef[slot * ROWP + e] = cv;
        if (cv != 0.0) atomicOr(&s_nz[k], 1u << (e / (NC * NC)));
      }
    }
  }
  __syncthreads();
  mbar_wait(bar, 0);
  if (live) {
    const int E01 = E0 * E1, EC = E01 * E2;
    const double* const nb = s_box + (ix - xs) + E0 * (iy - ys) + E01 * (lz - zs);   // this node in the box, component 0
    const double* cf = slots_ok ? s_coef + __popc(cmask & ((1u << cls) - 1u)) * ROWP : coef + (size_t)cls * ROW;
    const unsigned nz = slots_ok ? s_nz[cls] : 0x7fffu;
    const bool f2 = CHEBY && a.first2;
    double acc[NC] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int k = 0; k < PDE_NOFF; ++k) {
      if (!((nz >> k) & 1u)) continue;
      const int off = kOffDcomp(k, 0) + E0 * kOffDcomp(k, 1) + E01 * kOffDcomp(k, 2);
      double xk[NC];
#pragma unroll
      for (int j = 0; j < NC; ++j) xk[j] = nb[off + j * EC];
      if (f2) {   // the box holds the right-hand side: x1 = s0 D^-1 b with the class diagonal of the neighbour
        const int jx = ix + kOffDcomp(k, 0), jy = iy + kOffDcomp(k, 1), jz = lz + g.z0 + kOffDcomp(k, 2);
        const bool in = jx >= 0 && jx < g.nn[0] && jy >= 0 && jy < g.nn[1] && jz >= 0 && jz < g.nzg;
        const int ck = in ? node_class(g, jx, jy, jz) : 13;
#pragma unroll
        for (int j = 0; j < NC; ++j) xk[j] *= a.s0 * s_dinv[ck * NC + j];
      }
#pragma unroll
      for (int i = 0; i < NC; ++i)
#pragma unroll
        for (int j = 0; j < NC; ++j) acc[i] = fma(cf[k * NC * NC + i * NC + j], xk[j], acc[i]);
    }
    const double ld = a.b ? 0.0 : __ldg(load + cls);
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const double xo = nb[i * EC];
      const double B = a.b ? bv[i] : a.bconst[i] * ld;
      if (f2) {
        const double x1 = a.s0 * s_dinv[cls * NC + i] * xo;
        (a.y + i * g.comp_stride)[idxl] = fma(1.0 + a.c1, x1, a.c2 * s_dinv[cls * NC + i] * (xo - acc[i]));
      } else if (CHEBY) {
        const double di = __ldg(dinv + cls * NC + i);
        const double dprev = a.prev_mode == 1 ? xo - pv[i]
                           : (a.prev_mode == 2 ? xo : (a.prev_mode == 3 ? xo - a.s0 * di * B : 0.0));
        const double dn = a.c1 * dprev + a.c2 * di * (B - acc[i]);
        const double yv = xo + dn;
        (a.y + i * g.comp_stride)[idxl] = yv;
        acc_xy = fma(B, yv, acc_xy);
      } else {
        const double yv = a.bscale * B + a.ascale * acc[i];
        if (a.y) (a.y + i * g.comp_stride)[idxl] = yv;
        acc_xy = fma(xo, yv, acc_xy);
        acc_yy = fma(yv, yv, acc_yy);
      }
    }
  }
  if (a.do_reduce && a.defer) {
    __shared__ double sm2[2][FACE_NT / 32];
    double vv[2] = {acc_xy, acc_yy};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) vv[i] += __shfl_down_sync(0xffffffffu, vv[i], o);
      if ((threadIdx.x & 31) == 0) sm2[i][threadIdx.x >> 5] = vv[i];
    }
    __syncthreads();
    if (threadIdx.x < 2) {
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < FACE_NT / 32; ++w) t += sm2[threadIdx.x][w];
      a.defer[(size_t)blockIdx.x * RED_MAX_VALS + threadIdx.x] = t;
    }
  } else if (a.do_reduce) {
    if (CHEBY) {
      double vv[1] = {acc_xy};
      block_reduce_finalize<1, true>(vv, red, red_out);
    } else {
      double vv[2] = {acc_xy, acc_yy};
      block_reduce_finalize<2, true>(vv, red, red_out);
    }
  }
}

int launch_face_rows(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a, int* defer_blocks) {
  if (defer_blocks) *defer_blocks = 0;
  // fused first sweeps (cheby == 2): x1 = s0 D^-1 b needs the class diagonal of every neighbour, so the layer NEXT to a
  // natural face is computed here as well (two layers); only the 3-D kernel with the cached class table implements it
  const int layers = a.cheby == 2 ? 2 : 1;
  if (layers == 2 && (bc.side_excl || g.dim != 3 || a.reduce_slot_xy >= 0))
    PDE_FAIL("fused first sweeps on natural faces need a 3-D operator without the other_faces rule and no reduction");
  FaceSet fs;
  memset(&fs, 0, sizeof(fs));
  long long ntiles = 0;
  const int n0 = g.nn[0], n1 = g.nn[1];
  auto add = [&](int axis, int fixed, int lo0, int c0, int lo1, int c1) {
    if (c0 <= 0 || c1 <= 0 || fs.nface >= 12) return;
    const int f = fs.nface++;
    fs.axis[f] = axis; fs.fixed[f] = fixed;
    fs.lo[f][0] = lo0; fs.cnt[f][0] = c0; fs.lo[f][1] = lo1; fs.cnt[f][1] = c1;
    fs.tiles0[f] = (c0 + FACE_TU - 1) / FACE_TU;
    ntiles += (long long)fs.tiles0[f] * ((c1 + FACE_TV - 1) / FACE_TV);
    fs.tstart[f + 1] = (int)(ntiles > RED_MAX_BLOCKS ? RED_MAX_BLOCKS + 1LL : ntiles);
  };
  // a face whose Dirichlet flag is set contributes no free rows, except that the reference's "other_faces"
  // rule (side_excl) leaves the x-end columns of side faces free: keep such faces listed
  const bool keep_all = bc.side_excl != 0;
  const bool nat[6] = {!bc.on[0] || keep_all, !bc.on[1] || keep_all, !bc.on[2] || keep_all,
                       !bc.on[3] || keep_all, !bc.on[4] || keep_all, !bc.on[5] || keep_all};
  // nodes already taken by the x layers (y, z sets) and by the y layers (z sets)
  const int xl = (layers == 2 && nat[0]) ? 2 : 1, xh = (layers == 2 && nat[1]) ? n0 - 3 : n0 - 2;
  const int yl = g.nc[1] > 0 ? ((layers == 2 && nat[2]) ? 2 : 1) : 0;
  const int yh = g.nc[1] > 0 ? ((layers == 2 && nat[3]) ? n1 - 3 : n1 - 2) : 0;
  for (int ly = 0; ly < layers; ++ly) {
    if (g.nc[0] > 0 && n0 > 2 * ly) {
      if (nat[0]) add(0, ly, 0, n1, 0, g.nzl);
      if (nat[1]) add(0, n0 - 1 - ly, 0, n1, 0, g.nzl);
    }
    if (g.nc[1] > 0 && n1 > 2 * ly) {
      if (nat[2]) add(1, ly, xl, xh - xl + 1, 0, g.nzl);
      if (nat[3]) add(1, n1 - 1 - ly, xl, xh - xl + 1, 0, g.nzl);
    }
    if (g.nc[2] > 0 && (n1 > 2 || g.nc[1] == 0)) {
      const int zlo = ly - g.z0, zhi = g.nzg - 1 - ly - g.z0;          // local planes of the two layers
      if (nat[4] && zlo >= 0 && zlo < g.nzl) add(2, zlo, xl, xh - xl + 1, yl, yh - yl + 1);
      if (nat[5] && zhi >= 0 && zhi < g.nzl && zhi != zlo) add(2, zhi, xl, xh - xl + 1, yl, yh - yl + 1);
    }
  }
  if (ntiles == 0) return 0;
  if (ntiles > RED_MAX_BLOCKS) PDE_FAIL("face grid exceeds the reduction buffer");
  StencilDev sd;
  sd.x = a.x; sd.b = a.b; sd.y = a.y; sd.xprev = a.xprev; sd.prev_mode = a.prev_mode;
  for (int i = 0; i < 3; ++i) sd.bconst[i] = a.bconst[i];
  sd.bscale = a.bscale; sd.ascale = a.ascale; sd.c1 = a.c1; sd.c2 = a.c2; sd.s0 = a.s0;
  sd.do_reduce = a.reduce_slot_xy >= 0;
  sd.first2 = a.cheby == 2;
  sd.defer = (defer_blocks && sd.do_reduce) ? c->face_partials : nullptr;
  const int blocks = (int)ntiles;
  if (sd.defer) *defer_blocks = blocks;
  bool full = g.dim == 3 && g.nk == PDE_NOFF && g.comp_stride * op.ncomp < (1LL << 31);
  for (int k = 0; full && k < PDE_NOFF; ++k) full = g.kidx[k] == k;
  if (layers == 2 && !full) PDE_FAIL("fused first sweeps on natural faces: grid too large for the 3-D face kernel");
  double* out = sd.do_reduce ? c->scal + a.reduce_slot_xy : nullptr;
  if (full && op.ncomp == 3) {
    CUtensorMap t0, t1, t2;
    PDE_OK(field_tensor_map(a.x, g, 3, 4, FACE_TU + 2, &t0, FACE_TV + 2));
    PDE_OK(field_tensor_map(a.x, g, 3, FACE_TU + 4, 3, &t1, FACE_TV + 2));
    PDE_OK(field_tensor_map(a.x, g, 3, FACE_TU + 4, FACE_TV + 2, &t2, 3));
    static bool attr = false;
    if (!attr) {
      CUDA_OK(cudaFuncSetAttribute(k_face_tile<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_BOX * 8));
      CUDA_OK(cudaFuncSetAttribute(k_face_tile<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_BOX * 8));
      attr = true;
    }
    if (a.cheby) k_face_tile<true><<<blocks, FACE_NT, FT_BOX * 8, c->stream>>>(t0, t1, t2, g, bc, fs, op.coef, op.dinv, op.load, sd, c->red, out);
    else k_face_tile<false><<<blocks, FACE_NT, FT_BOX * 8, c->stream>>>(t0, t1, t2, g, bc, fs, op.coef, op.dinv, op.load, sd, c->red, out);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    return 0;
  }
#define FACE_LAUNCH(CH, FU)                                                                                      \
  DISPATCH_NC(op.ncomp, (k_face_rows<NC, CH, FU><<<blocks, FACE_NT, 0, c->stream>>>(g, bc, fs, op.coef, op.dinv, op.load, \
                                                                               sd, c->red, out)))
  if (a.cheby) {
    if (full) { FACE_LAUNCH(true, true); } else { FACE_LAUNCH(true, false); }
  } else {
    if (full) { FACE_LAUNCH(false, true); } else { FACE_LAUNCH(false, false); }
  }
#undef FACE_LAUNCH
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// GMG-PCG variants of the two vector updates: no class-dependent Jacobi diagonal is involved, so they run flat
// over the padded storage with 16-byte accesses (pads and ghost planes hold zeros in p, q, z and stay zero).
__global__ void __launch_bounds__(256)
k_cg_update_flat(double* __restrict__ x, double* __restrict__ r, const double* __restrict__ p,
                 const double* __restrict__ q, long long n, int ncomp, long long cs, const double* __restrict__ scal,
                 int s_rho, int s_pap, ReduceBuf red, double* out_rho_new) {
  const double pap = scal[s_pap], rho = scal[s_rho];
  const double alpha = pap > 0.0 ? rho / pap : 0.0;
  const long long n2 = n >> 1;
  double rr = 0.0;
  for (int cidx = 0; cidx < ncomp; ++cidx) {
    double2* x2 = reinterpret_cast<double2*>(x + cidx * cs);
    double2* r2 = reinterpret_cast<double2*>(r + cidx * cs);
    const double2* p2 = reinterpret_cast<const double2*>(p + cidx * cs);
    const double2* q2 = reinterpret_cast<const double2*>(q + cidx * cs);
    if (x == nullptr) {  // the x update rides on the p update of the same iteration (k_cg_pupdate_flat)
      for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
        const double2 qv = q2[i];
        double2 rv = r2[i];
        rv.x = fma(-alpha, qv.x, rv.x);
        rv.y = fma(-alpha, qv.y, rv.y);
        r2[i] = rv;
        rr = fma(rv.x, rv.x, rr);
        rr = fma(rv.y, rv.y, rr);
      }
      continue;
    }
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
      const double2 pv = p2[i], qv = q2[i];
      double2 xv = x2[i], rv = r2[i];
      xv.x = fma(alpha, pv.x, xv.x);
      xv.y = fma(alpha, pv.y, xv.y);
      rv.x = fma(-alpha, qv.x, rv.x);
      rv.y = fma(-alpha, qv.y, rv.y);
      x2[i] = xv;
      r2[i] = rv;
      rr = fma(rv.x, rv.x, rr);
      rr = fma(rv.y, rv.y, rr);
    }
  }
  // slots (rho_new, rr): the preconditioned product is filled in later by the V-cycle's last sweep
  double v[2] = {0.0, rr};
  block_reduce_finalize<2>(v, red, out_rho_new);
}

__global__ void __launch_bounds__(256)
k_cg_pupdate_flat(double* __restrict__ p, const double* __restrict__ z, long long n, int ncomp, long long cs,
                  const double* __restrict__ scal, int s_rho, int s_rho_new, int first, double* __restrict__ x,
                  int s_pap) {
  double beta = 0.0;
  if (!first) {
    const double rho = scal[s_rho];
    beta = rho > 0.0 ? scal[s_rho_new] / rho : 0.0;
  }
  const long long n2 = n >> 1;
  if (x != nullptr && !first) {
    // deferred x update of this iteration, x += alpha p_old, on the way (p is read here anyway: 8 B/dof less
    // traffic per iteration than updating x together with r)
    const double pap = scal[s_pap], rho = scal[s_rho];
    const double alpha = pap > 0.0 ? rho / pap : 0.0;
    for (int cidx = 0; cidx < ncomp; ++cidx) {
      double2* p2 = reinterpret_cast<double2*>(p + cidx * cs);
      double2* x2 = reinterpret_cast<double2*>(x + cidx * cs);
      if (z == nullptr) {   // the converged iteration: x += alpha p alone, p is not needed any more
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
          const double2 pv = p2[i];
          double2 xv = x2[i];
          xv.x = fma(alpha, pv.x, xv.x);
          xv.y = fma(alpha, pv.y, xv.y);
          x2[i] = xv;
        }
        continue;
      }
      const double2* z2 = reinterpret_cast<const double2*>(z + cidx * cs);
      for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
        const double2 zv = z2[i];
        double2 pv = p2[i], xv = x2[i];
        xv.x = fma(alpha, pv.x, xv.x);
        xv.y = fma(alpha, pv.y, xv.y);
        pv.x = fma(beta, pv.x, zv.x);
        pv.y = fma(beta, pv.y, zv.y);
        x2[i] = xv;
        p2[i] = pv;
      }
    }
    return;
  }
  for (int cidx = 0; cidx < ncomp; ++cidx) {
    double2* p2 = reinterpret_cast<double2*>(p + cidx * cs);
    const double2* z2 = reinterpret_cast<const double2*>(z + cidx * cs);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
      const double2 zv = z2[i];
      double2 pv = first ? make_double2(0.0, 0.0) : p2[i];
      pv.x = fma(beta, pv.x, zv.x);
      pv.y = fma(beta, pv.y, zv.y);
      p2[i] = pv;
    }
  }
}

int launch_cg_update(pde_ctx* c, const Grid& g, const OpDev& op, double* x, double* r, const double* p,
                     const double* q, int slot_rho, int slot_pap, int slot_rho_new, int slot_rr, int jacobi) {
  if (slot_rr != slot_rho_new + 1) PDE_FAIL("cg_update needs adjacent (rho_new, rr) slots");
  if (!jacobi) {
    int blocks = flat_blocks(c, g.total / 2, 256 * 2);
    k_cg_update_flat<<<blocks, 256, 0, c->stream>>>(x, r, p, q, g.total, op.ncomp, g.comp_stride, c->scal, slot_rho,
                                                    slot_pap, c->red, c->scal + slot_rho_new);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    return 0;
  }
  RowLaunch rl = row_launch(c, g);
  DISPATCH_NC(op.ncomp, (k_cg_update<NC><<<rl.grid, rl.block, 0, c->stream>>>(
                            g, op.dinv, x, r, p, q, c->scal, slot_rho, slot_pap, c->red, c->scal + slot_rho_new,
                            c->scal + slot_rr)));
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int launch_cg_pupdate(pde_ctx* c, const Grid& g, const OpDev& op, double* p, const double* r_or_z, int slot_rho,
                      int slot_rho_new, int first, int jacobi, double* x_deferred, int slot_pap) {
  if (!jacobi) {
    int blocks = flat_blocks(c, g.total / 2, 256 * 2);
    k_cg_pupdate_flat<<<blocks, 256, 0, c->stream>>>(p, r_or_z, g.total, op.ncomp, g.comp_stride, c->scal, slot_rho,
                                                     slot_rho_new, first, x_deferred, slot_pap);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    return 0;
  }
  RowLaunch rl = row_launch(c, g);
  DISPATCH_NC(op.ncomp, (k_cg_pupdate<NC><<<rl.grid, rl.block, 0, c->stream>>>(
                            g, op.dinv, p, r_or_z, c->scal, slot_rho, slot_rho_new, first, jacobi)));
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// ----------------------------------------------------------------------------------------------
// flat vector kernels over the padded range (pads are zero and stay zero)
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_dot(const double* __restrict__ a, const double* __restrict__ b, long long n, int ncomp, long long cs,
      ReduceBuf red, double* out) {
  double s = 0.0;
  const long long n2 = n >> 1;
  for (int cidx = 0; cidx < ncomp; ++cidx) {
    const double2* a2 = reinterpret_cast<const double2*>(a + cidx * cs);
    const double2* b2 = reinterpret_cast<const double2*>(b + cidx * cs);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
      const double2 u = a2[i], w = b2[i];
      s = fma(u.x, w.x, s);
      s = fma(u.y, w.y, s);
    }
  }
  double v[1] = {s};
  block_reduce_finalize<1>(v, red, out);
}

__global__ void __launch_bounds__(256)
k_axpy(double* __restrict__ y, const double* __restrict__ x, double alpha, long long n, int ncomp, long long cs,
       int mode) {
  const long long n2 = n >> 1;
  for (int cidx = 0; cidx < ncomp; ++cidx) {
    double2* y2 = reinterpret_cast<double2*>(y + cidx * cs);
    const double2* x2 = reinterpret_cast<const double2*>(x + cidx * cs);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
      if (mode == 0) {  // y += alpha x
        double2 u = y2[i];
        const double2 w = x2[i];
        u.x = fma(alpha, w.x, u.x);
        u.y = fma(alpha, w.y, u.y);
        y2[i] = u;
      } else if (mode == 1) {  // y = x
        y2[i] = x2[i];
      } else {  // y = 0
        y2[i] = make_double2(0.0, 0.0);
      }
    }
  }
}

int launch_dot(pde_ctx* c, const Grid& g, int ncomp, const double* a, const double* b, int slot) {
  int blocks = flat_blocks(c, g.total / 2, 256 * 4);
  k_dot<<<blocks, 256, 0, c->stream>>>(a, b, g.total, ncomp, g.comp_stride, c->red, c->scal + slot);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
static int launch_axpy_mode(pde_ctx* c, const Grid& g, int ncomp, double* y, const double* x, double alpha, int mode) {
  int blocks = flat_blocks(c, g.total / 2, 256 * 4);
  k_axpy<<<blocks, 256, 0, c->stream>>>(y, x, alpha, g.total, ncomp, g.comp_stride, mode);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_zero(pde_ctx* c, const Grid& g, int ncomp, double* a) { return launch_axpy_mode(c, g, ncomp, a, a, 0.0, 2); }
int launch_copy(pde_ctx* c, const Grid& g, int ncomp, double* dst, const double* src) {
  return launch_axpy_mode(c, g, ncomp, dst, src, 0.0, 1);
}
int launch_axpy(pde_ctx* c, const Grid& g, int ncomp, double* y, const double* x, double alpha) {
  return launch_axpy_mode(c, g, ncomp, y, x, alpha, 0);
}

// ----------------------------------------------------------------------------------------------
// multigrid transfer + first Chebyshev sweep
// ----------------------------------------------------------------------------------------------
template <int NC>
__global__ void __launch_bounds__(128)
k_cheby_first(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc, const double* __restrict__ dinv,
              const double* b, double* x, double s) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const int gz = lz + g.z0;
    const long long rbase = (long long)g.PX * iy + g.plane * lz;
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      double bcv;
      const bool isdir = bc_node(g, bc, ix, iy, gz, &bcv);
      const int cls = node_class(g, ix, iy, gz);
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const long long ii = rbase + ix + i * g.comp_stride;
        x[ii] = isdir ? 0.0 : s * __ldg(dinv + cls * NC + i) * b[ii];
      }
    }
  }
}

int launch_cheby_first(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const double* b, double* x,
                       double s) {
  RowLaunch rl = row_launch(c, g);
  DISPATCH_NC(op.ncomp, (k_cheby_first<NC><<<rl.grid, rl.block, 0, c->stream>>>(g, bc, op.dinv, b, x, s)));
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// R = P^T : coarse node C gathers r_f(2C) + 1/2 sum over the 14 (6, 2) Kuhn edge directions
template <int NC>
__global__ void __launch_bounds__(256)
k_restrict(const __grid_constant__ Grid gf, const __grid_constant__ Grid gc, const __grid_constant__ BcDev bcc,
           const double* __restrict__ rf, double* __restrict__ bc_out) {
  // flat over the coarse nodes (a row-per-block mapping idles a sixth of the threads on 641-node rows), 32-bit index
  // arithmetic while the level is small enough
  const unsigned n0 = (unsigned)gc.nn[0], n1 = (unsigned)gc.nn[1];
  const long long total = (long long)n0 * n1 * gc.nzl;
  const bool small = total < (1LL << 32);
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const unsigned row = small ? (unsigned)t / n0 : (unsigned)(t / n0);
    const int ix = (int)(t - (long long)row * n0);
    const int iy = (int)(row % n1);
    const int lz = (int)(row / n1);
    const int gz = lz + gc.z0;
    const long long cbase = (long long)gc.PX * iy + gc.plane * lz;
    const int fy = gf.nc[1] > 0 ? 2 * iy : 0;
    const int flz = (gf.nc[2] > 0 ? 2 * gz : 0) - gf.z0;
    const long long fi = (long long)gf.PX * fy + gf.plane * flz + 2 * ix;
    double bcv;
    const bool isdir = bc_node(gc, bcc, ix, iy, gz, &bcv);
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      double s = 0.0;
      if (!isdir) {
        const double* rp = rf + i * gf.comp_stride;
        double nb = 0.0;
        for (int k = 1; k < gf.nk; ++k) nb += rp[fi + gf.koff[k]];
        s = rp[fi] + 0.5 * nb;
      }
      bc_out[cbase + ix + i * gc.comp_stride] = s;
    }
  }
}

int launch_restrict(pde_ctx* c, const Grid& gf, const Grid& gc, const BcDev& bcc, int ncomp, const double* rf,
                    double* bcoarse) {
  const int blocks = flat_blocks(c, (long long)gc.nn[0] * gc.nn[1] * gc.nzl, 256);
  DISPATCH_NC(ncomp, (k_restrict<NC><<<blocks, 256, 0, c->stream>>>(gf, gc, bcc, rf, bcoarse)));
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// x_f += P x_c : fine node with parity pi is the midpoint of the coarse Kuhn edge ((f-pi)/2,(f+pi)/2)
template <int NC>
__global__ void __launch_bounds__(256)
k_prolong_add(const __grid_constant__ Grid gf, const __grid_constant__ Grid gc, const __grid_constant__ BcDev bcf,
              const double* __restrict__ xc, double* __restrict__ xf, int ghost) {
  // flat over (row, node pair): two nodes (even ix, ix + 1) per thread, one 16-byte read-modify-write of the fine row
  // and three coarse values (rows start 32-byte aligned; the node after the last one of a row is a pad column, which
  // is written back unchanged).  A row-per-block mapping idles a third of the threads on 513-node rows.
  const int nzr = gf.nzl + 2 * ghost;
  const unsigned npair = (unsigned)(gf.nn[0] + 1) / 2;
  const long long total = (long long)gf.nn[1] * nzr * npair;
  const bool small = total < (1LL << 32);   // 32-bit index arithmetic (a 64-bit division costs ~100 instructions per pair)
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const unsigned row = small ? (unsigned)t / npair : (unsigned)(t / npair);
    const int k = (int)(t - (long long)row * npair);
    const int iy = (int)(row % (unsigned)gf.nn[1]);
    const int lz = (int)(row / (unsigned)gf.nn[1]) - ghost;
    const int gz = lz + gf.z0;
    if (gz < 0 || gz > gf.nzg - 1) continue;   // ghost plane beyond the domain end
    const int ix = 2 * k;
    double bcv;
    const bool f0 = !bc_node(gf, bcf, ix, iy, gz, &bcv);
    const bool f1 = ix + 1 < gf.nn[0] && !bc_node(gf, bcf, ix + 1, iy, gz, &bcv);
    if (!f0 && !f1) continue;
    const long long fbase = (long long)gf.PX * iy + gf.plane * lz;
    const int py = gf.nc[1] > 0 ? (iy & 1) : 0;
    const int pz = gf.nc[2] > 0 ? (gz & 1) : 0;
    const int cy = gf.nc[1] > 0 ? (iy - py) / 2 : 0;
    const int clz = (gf.nc[2] > 0 ? (gz - pz) / 2 : 0) - gc.z0;
    const long long lo = (long long)gc.PX * cy + gc.plane * clz + k;
    const long long cpy = (long long)gc.PX * py + gc.plane * pz;
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const double* cp = xc + i * gc.comp_stride;
      double2* fp = reinterpret_cast<double2*>(xf + fbase + ix + i * gf.comp_stride);
      double2 v = *fp;
      const double c0 = cp[lo];
      if (f0) v.x += 0.5 * (c0 + cp[lo + cpy]);
      if (f1) v.y += 0.5 * (c0 + cp[lo + 1 + cpy]);
      *fp = v;
    }
  }
}

int launch_prolong_add(pde_ctx* c, const Grid& gf, const Grid& gc, const BcDev& bcf, int ncomp, const double* xc,
                       double* xf, int ghost) {
  const long long total = (long long)gf.nn[1] * (gf.nzl + 2 * ghost) * ((gf.nn[0] + 1) / 2);
  if (gf.nn[1] * (long long)(gf.nzl + 2 * ghost) >= (1LL << 32)) PDE_FAIL("prolongation: too many rows");
  const int blocks = flat_blocks(c, total, 256);
  DISPATCH_NC(ncomp, (k_prolong_add<NC><<<blocks, 256, 0, c->stream>>>(gf, gc, bcf, xc, xf, ghost)));
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// coarsest level: x = A^-1 b on the free dofs, one warp per row of the precomputed dense inverse
__global__ void __launch_bounds__(256)
k_dense_solve(int n, const double* __restrict__ Ainv, const long long* __restrict__ idx, const double* __restrict__ b,
              double* __restrict__ x) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  double s = 0.0;
  for (int j = lane; j < n; j += 32) s = fma(Ainv[(size_t)warp * n + j], b[idx[j]], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0) x[idx[warp]] = s;
}

int launch_dense_solve(pde_ctx* c, int n, const double* Ainv, const long long* idx, const double* b, double* x) {
  if (n <= 0) return 0;
  int blocks = (n * 32 + 255) / 256;
  k_dense_solve<<<blocks, 256, 0, c->stream>>>(n, Ainv, idx, b, x);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// multi-rank coarsest level: every rank holds the global dense inverse; the right-hand side is assembled
// by an all-reduce of the owned entries, each rank then computes the rows it owns
__global__ void __launch_bounds__(256)
k_dense_gather(int n, const long long* __restrict__ idx, const double* __restrict__ b, double* __restrict__ bglob) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) bglob[j] = idx[j] >= 0 ? b[idx[j]] : 0.0;
}
__global__ void __launch_bounds__(256)
k_dense_solve_owned(int n, const double* __restrict__ Ainv, const long long* __restrict__ idx,
                    const double* __restrict__ bglob, double* __restrict__ x) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n || idx[warp] < 0) return;
  double s = 0.0;
  for (int j = lane; j < n; j += 32) s = fma(Ainv[(size_t)warp * n + j], bglob[j], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0) x[idx[warp]] = s;
}
int launch_dense_gather(pde_ctx* c, int n, const long long* idx, const double* b, double* bglob) {
  if (n <= 0) return 0;
  k_dense_gather<<<(n + 255) / 256, 256, 0, c->stream>>>(n, idx, b, bglob);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_dense_solve_owned(pde_ctx* c, int n, const double* Ainv, const long long* idx, const double* bglob,
                             double* x) {
  if (n <= 0) return 0;
  k_dense_solve_owned<<<(n * 32 + 255) / 256, 256, 0, c->stream>>>(n, Ainv, idx, bglob, x);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// ----------------------------------------------------------------------------------------------
// fields: initial condition / BC values / dense <-> padded layout
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_fill_ic(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc, double* __restrict__ u, double value,
          int fill, int apply_bc) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const long long rbase = (long long)g.PX * iy + g.plane * lz;
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      double bcv;
      const bool isdir = apply_bc && bc_node(g, bc, ix, iy, lz + g.z0, &bcv);
      if (isdir) u[rbase + ix] = bcv;
      else if (fill) u[rbase + ix] = value;
    }
  }
}
// x_i = sin(0.37 i + comp) + 0.5 on free nodes, 0 on Dirichlet nodes (benchmarks, power iteration)
__global__ void __launch_bounds__(128)
k_fill_pattern(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc, int ncomp, double* __restrict__ x) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      double bcv;
      const bool isdir = bc_node(g, bc, ix, iy, lz + g.z0, &bcv);
      const long long node = ((long long)(lz + g.z0) * g.nn[1] + iy) * g.nn[0] + ix;
      for (int i = 0; i < ncomp; ++i)
        x[(long long)g.PX * iy + g.plane * lz + ix + i * g.comp_stride] =
            isdir ? 0.0 : sin(0.37 * (double)(node % 1000003) + i) + 0.5;
    }
  }
}
int launch_fill_pattern(pde_ctx* c, const Grid& g, const BcDev& bc, int ncomp, double* x) {
  RowLaunch rl = row_launch(c, g);
  k_fill_pattern<<<rl.grid, rl.block, 0, c->stream>>>(g, bc, ncomp, x);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// ghost planes after a halo exchange of `scale` * (the k_fill_pattern field without Dirichlet nodes): count the
// entries that differ from the value the owning neighbour holds (bitwise: the scale is a power of two)
__global__ void __launch_bounds__(128)
k_halo_verify(const __grid_constant__ Grid g, int ncomp, int depth, const double* __restrict__ x, double scale,
              unsigned long long* bad) {
  const long long rows = (long long)g.nn[1] * 2 * depth;
  unsigned long long nbad = 0;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int q = (int)(row / g.nn[1]);                         // 0..depth-1 below, depth..2*depth-1 above
    const int lz = q < depth ? -1 - q : g.nzl + (q - depth);
    const int gz = lz + g.z0;
    if (gz < 0 || gz > g.nzg - 1) continue;                     // no neighbour on that side
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const long long node = ((long long)gz * g.nn[1] + iy) * g.nn[0] + ix;
      for (int i = 0; i < ncomp; ++i) {
        const double want = scale * (sin(0.37 * (double)(node % 1000003) + i) + 0.5);
        if (x[(long long)g.PX * iy + g.plane * lz + ix + i * g.comp_stride] != want) ++nbad;
      }
    }
  }
  if (nbad) atomicAdd(bad, nbad);
}
int launch_halo_verify(pde_ctx* c, const Grid& g, int ncomp, int depth, const double* x, double scale,
                       unsigned long long* bad) {
  RowLaunch rl = row_launch(c, g);
  k_halo_verify<<<rl.grid, rl.block, 0, c->stream>>>(g, ncomp, depth, x, scale, bad);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int launch_fill_ic(pde_ctx* c, const Grid& g, const BcDev& bc, double* u, double value, int apply_bc) {
  RowLaunch rl = row_launch(c, g);
  k_fill_ic<<<rl.grid, rl.block, 0, c->stream>>>(g, bc, u, value, 1, apply_bc);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_apply_bc_values(pde_ctx* c, const Grid& g, const BcDev& bc, double* u) {
  RowLaunch rl = row_launch(c, g);
  k_fill_ic<<<rl.grid, rl.block, 0, c->stream>>>(g, bc, u, 0.0, 0, 1);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// dense = natural lattice order of the local planes; interleave: dense[node*nc+c] else dense[c*nloc+node]
template <bool PACK>
__global__ void __launch_bounds__(128)
k_pack(const __grid_constant__ Grid g, int ncomp, double* __restrict__ padded, double* __restrict__ dense,
       int interleave) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  const long long nloc = (long long)g.nn[0] * rows;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const long long rbase = (long long)g.PX * iy + g.plane * lz;
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const long long node = row * g.nn[0] + ix;
      for (int i = 0; i < ncomp; ++i) {
        const long long di = interleave ? node * ncomp + i : i * nloc + node;
        if (PACK) dense[di] = padded[rbase + ix + i * g.comp_stride];
        else padded[rbase + ix + i * g.comp_stride] = dense[di];
      }
    }
  }
}
int launch_pack(pde_ctx* c, const Grid& g, int ncomp, const double* padded, double* dense, int interleave) {
  RowLaunch rl = row_launch(c, g);
  k_pack<true><<<rl.grid, rl.block, 0, c->stream>>>(g, ncomp, const_cast<double*>(padded), dense, interleave);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_unpack(pde_ctx* c, const Grid& g, int ncomp, const double* dense, double* padded, int interleave) {
  RowLaunch rl = row_launch(c, g);
  k_pack<false><<<rl.grid, rl.block, 0, c->stream>>>(g, ncomp, padded, const_cast<double*>(dense), interleave);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// ----------------------------------------------------------------------------------------------
// load vector of project(eq_expr, Vs): b_i = sum over incident simplices of value_simplex*|simplex|/(d+1)
// gather form (no atomics, deterministic).  mode 0: von-Mises stress, 1: von-Mises strain,
// 2: axial strain du/dx, 3: axial stress E du/dx (1D bar).
// ----------------------------------------------------------------------------------------------
template <int NC>
__global__ void __launch_bounds__(128)
k_cell_rhs(const __grid_constant__ Grid g, const __grid_constant__ SimplexGeom sg, const double* __restrict__ u,
           double* __restrict__ rhs, int mode, double lam, double mu, double Emod) {
  // component i <-> internal axis axm[i]
  const int axm[3] = {0, g.dim == 2 ? 2 : 1, 2};
  const long long rows = (long long)g.nn[1] * g.nzl;
  const double w = sg.vol / (double)(g.dim + 1);
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const int gz = lz + g.z0;
    const long long rbase = (long long)g.PX * iy + g.plane * lz;
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      const long long idx = rbase + ix;
      double acc = 0.0;
      for (int o = 0; o < 8; ++o) {
        const int ox = o & 1, oy = (o >> 1) & 1, oz = (o >> 2) & 1;
        if ((ox && (g.nc[0] == 0 || ix == 0)) || (!ox && g.nc[0] > 0 && ix == g.nn[0] - 1)) continue;
        if ((oy && (g.nc[1] == 0 || iy == 0)) || (!oy && g.nc[1] > 0 && iy == g.nn[1] - 1)) continue;
        if ((oz && (g.nc[2] == 0 || gz == 0)) || (!oz && g.nc[2] > 0 && gz == g.nzg - 1)) continue;
        const long long cell0 = idx - ox - (long long)g.PX * oy - g.plane * oz;  // corner 0 of the cell
        for (int t = 0; t < sg.nsimp; ++t) {
          bool has = false;
          for (int a = 0; a < sg.nv; ++a) has |= (sg.corner[t][a] == o);
          if (!has) continue;
          double gu[NC][3];
#pragma unroll
          for (int i = 0; i < NC; ++i) gu[i][0] = gu[i][1] = gu[i][2] = 0.0;
          for (int a = 0; a < sg.nv; ++a) {
            const int cb = sg.corner[t][a];
            const long long vi = cell0 + (cb & 1) + (long long)g.PX * ((cb >> 1) & 1) + g.plane * ((cb >> 2) & 1);
#pragma unroll
            for (int i = 0; i < NC; ++i) {
              const double uv = u[vi + i * g.comp_stride];
              gu[i][0] = fma(uv, sg.G[t][a][0], gu[i][0]);
              gu[i][1] = fma(uv, sg.G[t][a][1], gu[i][1]);
              gu[i][2] = fma(uv, sg.G[t][a][2], gu[i][2]);
            }
          }
          double val;
          if (mode >= 2) {
            val = gu[0][0] * (mode == 3 ? Emod : 1.0);
          } else {
            double eps[NC][NC];
            double tr = 0.0;
#pragma unroll
            for (int i = 0; i < NC; ++i) {
#pragma unroll
              for (int j = 0; j < NC; ++j) eps[i][j] = 0.5 * (gu[i][axm[j]] + gu[j][axm[i]]);
              tr += eps[i][i];
            }
            double ss = 0.0;
            if (mode == 1) {
#pragma unroll
              for (int i = 0; i < NC; ++i)
#pragma unroll
                for (int j = 0; j < NC; ++j) {
                  const double dv = eps[i][j] - (i == j ? (1.0 / 3.0) * tr : 0.0);
                  ss = fma(dv, dv, ss);
                }
              val = sqrt(2.0 / 3.0 * ss);
            } else {
              double trs = 0.0;
              double sig[NC][NC];
#pragma unroll
              for (int i = 0; i < NC; ++i) {
#pragma unroll
                for (int j = 0; j < NC; ++j) sig[i][j] = 2.0 * mu * eps[i][j] + (i == j ? lam * tr : 0.0);
                trs += sig[i][i];
              }
#pragma unroll
              for (int i = 0; i < NC; ++i)
#pragma unroll
                for (int j = 0; j < NC; ++j) {
                  const double dv = sig[i][j] - (i == j ? (1.0 / 3.0) * trs : 0.0);
                  ss = fma(dv, dv, ss);
                }
              val = sqrt(3.0 / 2.0 * ss);
            }
          }
          acc = fma(val, w, acc);
        }
      }
      rhs[idx] = acc;
    }
  }
}

// ---- 3-D von Mises load vector in two passes ---------------------------------------------------------------------
// k_cell_rhs evaluates the 24 simplices around every node (each simplex four times over, with table-driven gradients):
// 29.6 ms at config 5, 60x off its traffic.  The 3-D path computes every Kuhn simplex ONCE per cell (k_cell_vm: three
// edge differences per component give the displacement gradient of the path simplex 0 -> e_a -> e_a+e_b -> (1,1,1)) and
// leaves, per cell, the sum of the values of the simplices that contain each of its corners (7 planes of doubles, SoA;
// corners 0 and 7 are in all six); k_cell_gather then adds the (up to) eight cell-corner sums of a node in fixed order.
__device__ __forceinline__ double vm_value(const double (&gu)[3][3], int mode, double lam, double mu) {
  double eps[3][3];
  double tr = 0.0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 3; ++j) eps[i][j] = 0.5 * (gu[i][j] + gu[j][i]);
    tr += eps[i][i];
  }
  double ss = 0.0;
  if (mode == 1) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const double dv = eps[i][j] - (i == j ? (1.0 / 3.0) * tr : 0.0);
        ss = fma(dv, dv, ss);
      }
    return sqrt(2.0 / 3.0 * ss);
  }
  double trs = 0.0, sig[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 3; ++j) sig[i][j] = 2.0 * mu * eps[i][j] + (i == j ? lam * tr : 0.0);
    trs += sig[i][i];
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double dv = sig[i][j] - (i == j ? (1.0 / 3.0) * trs : 0.0);
      ss = fma(dv, dv, ss);
    }
  return sqrt(3.0 / 2.0 * ss);
}

// cells: x fastest, then y, then local cell layer lz - lzmin (the layer below local plane 0 uses the lower halo plane)
__global__ void __launch_bounds__(256)
k_cell_vm(const __grid_constant__ Grid g, const double* __restrict__ u, double* __restrict__ S, long long ncells, int lzmin,
          int mode, double lam, double mu) {
  const double ih[3] = {1.0 / g.h[0], 1.0 / g.h[1], 1.0 / g.h[2]};
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < ncells; t += (long long)gridDim.x * blockDim.x) {
    const int cx = (int)(t % g.nc[0]);
    const long long r = t / g.nc[0];
    const int cy = (int)(r % g.nc[1]);
    const int lz = (int)(r / g.nc[1]) + lzmin;
    const long long base = (long long)g.PX * cy + g.plane * lz + cx;
    double uc[8][3];   // corner o = ox + 2 oy + 4 oz
#pragma unroll
    for (int o = 0; o < 8; ++o)
#pragma unroll
      for (int i = 0; i < 3; ++i)
        uc[o][i] = u[base + (o & 1) + (long long)g.PX * ((o >> 1) & 1) + g.plane * ((o >> 2) & 1) + i * g.comp_stride];
    double Sv[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) Sv[o] = 0.0;
    // the six Kuhn simplices: path 0 -> e_a -> e_a + e_b -> 7 for the permutations (a, b, c)
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      constexpr int P[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};
      const int a = P[p][0], b = P[p][1], cc = P[p][2];
      const int v1 = 1 << a, v2 = v1 | (1 << b);
      double gu[3][3];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        gu[i][a] = (uc[v1][i] - uc[0][i]) * ih[a];
        gu[i][b] = (uc[v2][i] - uc[v1][i]) * ih[b];
        gu[i][cc] = (uc[7][i] - uc[v2][i]) * ih[cc];
      }
      const double val = vm_value(gu, mode, lam, mu);
      Sv[0] += val; Sv[v1] += val; Sv[v2] += val;
    }
#pragma unroll
    for (int o = 0; o < 7; ++o) S[(long long)o * ncells + t] = Sv[o];   // corner 7 = corner 0: every simplex has both
  }
}

__global__ void __launch_bounds__(256)
k_cell_gather(const __grid_constant__ Grid g, const double* __restrict__ S, double* __restrict__ rhs, long long ncells,
              int lzmin, int lzmax, double w, int pa, int pb) {
  // node planes [pa, pb); S holds the cell layers lzmin .. lzmax (layers outside the domain are simply not listed)
  const long long nodes = (long long)g.nn[0] * g.nn[1] * (pb - pa);
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < nodes; t += (long long)gridDim.x * blockDim.x) {
    const int ix = (int)(t % g.nn[0]);
    const long long r = t / g.nn[0];
    const int iy = (int)(r % g.nn[1]);
    const int lz = (int)(r / g.nn[1]) + pa;
    double acc = 0.0;
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      const int cx = ix - (o & 1), cy = iy - ((o >> 1) & 1), cz = lz - ((o >> 2) & 1);
      if (cx < 0 || cx >= g.nc[0] || cy < 0 || cy >= g.nc[1] || cz < lzmin || cz > lzmax) continue;
      const long long cell = cx + (long long)g.nc[0] * (cy + (long long)g.nc[1] * (cz - lzmin));
      acc += S[(long long)(o == 7 ? 0 : o) * ncells + cell];
    }
    rhs[(long long)g.PX * iy + g.plane * lz + ix] = w * acc;
  }
}

// is the simplex table the Kuhn split (every simplex a path 0 -> e_a -> e_a + e_b -> 7)?
static bool kuhn_split(const SimplexGeom& sg) {
  if (sg.nsimp != 6 || sg.nv != 4) return false;
  unsigned seen = 0;
  for (int t = 0; t < 6; ++t) {
    unsigned set = 0;
    for (int a = 0; a < 4; ++a) set |= 1u << sg.corner[t][a];
    if (!(set & 1u) || !(set & 128u) || __builtin_popcount(set) != 4) return false;
    int v1 = -1, v2 = -1;
    for (int o = 1; o < 7; ++o)
      if (set & (1u << o)) { if (__builtin_popcount((unsigned)o) == 1) v1 = o; else v2 = o; }
    if (v1 < 0 || v2 < 0 || (v1 & v2) != v1) return false;
    seen |= 1u << (v1 * 8 + v2) % 32;
  }
  return __builtin_popcount(seen) == 6;
}

int launch_cell_rhs(pde_ctx* c, const Grid& g, int ncomp, const SimplexGeom& sg, const double* u, double* rhs,
                    int mode, double lam, double mu, double Emod) {
  static const int two_pass = getenv("PDE_B200_CELL_2PASS") ? atoi(getenv("PDE_B200_CELL_2PASS")) : 1;
  if (two_pass && g.dim == 3 && ncomp == 3 && mode <= 1 && kuhn_split(sg) && g.nc[0] > 0 && g.nc[1] > 0 && g.nc[2] > 0) {
    // chunks of node planes, so that the cell-sum scratch stays small and cached on the context (a 4.7 GB allocation per
    // solve costs tens of milliseconds and, now and then, most of a second)
    const int gl0 = g.z0 > 0 ? -1 : 0;                                   // first / last cell layer this rank can form
    const int gl1 = (g.nzl - 1 > g.nzg - 2 - g.z0) ? g.nzg - 2 - g.z0 : g.nzl - 1;
    const long long per_layer = (long long)g.nc[0] * g.nc[1];
    int chunk = (int)((48LL << 20) / (per_layer > 0 ? per_layer : 1));   // about 48 M cells (2.7 GB / 7 planes -> 384 MB) at most
    chunk = chunk < 2 ? 2 : (chunk > 32 ? 32 : chunk);
    const size_t need = sizeof(double) * 7 * (size_t)per_layer * (chunk + 1);
    if (c->scratch_bytes < need) {
      if (c->scratch) { CUDA_OK(cudaStreamSynchronize(c->stream)); CUDA_OK(cudaFree(c->scratch)); c->scratch = nullptr; c->scratch_bytes = 0; }
      CUDA_OK(cudaMalloc(&c->scratch, need));
      c->scratch_bytes = need;
    }
    double* S = (double*)c->scratch;
    for (int pa = 0; pa < g.nzl; pa += chunk) {
      const int pb = pa + chunk < g.nzl ? pa + chunk : g.nzl;
      const int lzmin = pa - 1 < gl0 ? gl0 : pa - 1;                     // node plane p touches the cell layers p-1 and p
      const int lzmax = pb - 1 > gl1 ? gl1 : pb - 1;
      const long long ncells = per_layer * (lzmax - lzmin + 1);
      if (ncells > 0)
        k_cell_vm<<<flat_blocks(c, ncells, 256), 256, 0, c->stream>>>(g, u, S, ncells, lzmin, mode, lam, mu);
      k_cell_gather<<<flat_blocks(c, (long long)g.nn[0] * g.nn[1] * (pb - pa), 256), 256, 0, c->stream>>>(
          g, S, rhs, ncells > 0 ? ncells : 1, lzmin, lzmax, sg.vol / 4.0, pa, pb);
      c->launches += 2;
    }
    CUDA_OK(cudaGetLastError());
    return 0;
  }
  RowLaunch rl = row_launch(c, g);
  DISPATCH_NC(ncomp, (k_cell_rhs<NC><<<rl.grid, rl.block, 0, c->stream>>>(g, sg, u, rhs, mode, lam, mu, Emod)));
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// ----------------------------------------------------------------------------------------------
// load vector of project(Expression("A*cos(k x)[*cos(k y)[*cos(k z)]]", degree=2), V)   (:276-290, 408-421,
// 672-685): the expression is interpolated into P2 on every cell (values at vertices and edge midpoints)
// and integrated exactly against the P1 basis.  The expression is separable, so its values come from one
// table per axis sampled on the half-step lattice: tab[m] = trig(k * 0.5*(x[m/2] + x[(m+1)/2])).
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_trig_table(int dim, int n, double lo, double Ls, int use_sin, double kw, int len, double* __restrict__ tab) {
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < len; m += gridDim.x * blockDim.x) {
    const double ia = (double)(m / 2), ib = (double)((m + 1) / 2), dn = (double)n;
    double xa, xb;   // lo + ... with lo = 0 is exact, so the box-at-origin values are unchanged
    if (dim == 3) { xa = __dadd_rn(lo, __ddiv_rn(__dmul_rn(ia, Ls), dn)); xb = __dadd_rn(lo, __ddiv_rn(__dmul_rn(ib, Ls), dn)); }
    else { xa = __dadd_rn(lo, __dmul_rn(__ddiv_rn(Ls, dn), ia)); xb = __dadd_rn(lo, __dmul_rn(__ddiv_rn(Ls, dn), ib)); }
    const double x = 0.5 * (xa + xb);
    tab[m] = use_sin ? sin(kw * x) : cos(kw * x);
  }
}

struct P2Weights {
  double vself, voth, ein, eout;
};

__global__ void __launch_bounds__(128)
k_p2_load(const __grid_constant__ Grid g, const __grid_constant__ SimplexGeom sg, const __grid_constant__ P2Weights w,
          double amp, const double* __restrict__ tx, const double* __restrict__ ty, const double* __restrict__ tz,
          double* __restrict__ rhs) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    const int gz = lz + g.z0;
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      double acc = 0.0;
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
          // value at the point with doubled lattice index (mx,my,mz)
          auto val = [&](int ca, int cb) {
            const int mx = 2 * cx + (ca & 1) + (cb & 1);
            const int my = 2 * cy + ((ca >> 1) & 1) + ((cb >> 1) & 1);
            const int mz = 2 * cz + ((ca >> 2) & 1) + ((cb >> 2) & 1);
            double v = amp * tx[mx];
            if (g.nc[1] > 0) v *= ty[my];
            if (g.nc[2] > 0) v *= tz[mz];
            return v;
          };
          double s = 0.0;
          for (int a = 0; a < sg.nv; ++a) s = fma(val(sg.corner[t][a], sg.corner[t][a]), a == li ? w.vself : w.voth, s);
          for (int a = 0; a < sg.nv; ++a)
            for (int b = a + 1; b < sg.nv; ++b)
              s = fma(val(sg.corner[t][a], sg.corner[t][b]), (a == li || b == li) ? w.ein : w.eout, s);
          acc = fma(s, sg.vol, acc);
        }
      }
      rhs[(long long)g.PX * iy + g.plane * lz + ix] = acc;
    }
  }
}

int launch_p2_load(pde_ctx* c, const Grid& g, const SimplexGeom& sg, double amp, double kw, int use_sin,
                   const int32_t n_user[3], const double L_user[3], double* rhs, const double* lo_user) {
  // internal axis of user axis q: dim 2 maps user y -> internal z
  const int dim = g.dim;
  double* tabs[3] = {nullptr, nullptr, nullptr};
  int rc = 0;
  for (int q = 0; q < dim && !rc; ++q) {
    const int iax = (dim == 2 && q == 1) ? 2 : q;
    const int len = 2 * n_user[q] + 1;
    if (cudaMalloc(&tabs[iax], sizeof(double) * len) != cudaSuccess) { pde_set_error("cudaMalloc failed (trig table)"); rc = 1; break; }
    k_trig_table<<<(len + 255) / 256, 256, 0, c->stream>>>(dim, n_user[q], lo_user ? lo_user[q] : 0.0, L_user[q], use_sin, kw, len,
                                                           tabs[iax]);
    c->launches++;
  }
  if (!rc) {
    // int over the simplex of barycentric monomials: |c| d! prod(alpha!) / (d + |alpha|)!   (|c| applied in-kernel)
    auto fac = [](int k) { double f = 1; for (int i = 2; i <= k; ++i) f *= i; return f; };
    auto I = [&](int a, int b, int cc) { return fac(dim) * fac(a) * fac(b) * fac(cc) / fac(dim + a + b + cc); };
    P2Weights w;
    w.vself = 2 * I(3, 0, 0) - I(2, 0, 0);
    w.voth = 2 * I(2, 1, 0) - I(1, 1, 0);
    w.ein = 4 * I(2, 1, 0);
    w.eout = dim >= 2 ? 4 * I(1, 1, 1) : 0.0;
    RowLaunch rl = row_launch(c, g);
    // absent axes point at the x table (never multiplied in)
    k_p2_load<<<rl.grid, rl.block, 0, c->stream>>>(g, sg, w, amp, tabs[0], tabs[1] ? tabs[1] : tabs[0],
                                                   tabs[2] ? tabs[2] : tabs[0], rhs);
    c->launches++;
    if (cudaGetLastError() != cudaSuccess) { pde_set_error("k_p2_load launch failed"); rc = 1; }
  }
  cudaStreamSynchronize(c->stream);
  for (int q = 0; q < 3; ++q)
    if (tabs[q]) cudaFree(tabs[q]);
  return rc;
}

// ----------------------------------------------------------------------------------------------
// mesh / dof-map / boundary-set generation (bit-exact integer + FP64 coordinate expressions)
// ----------------------------------------------------------------------------------------------
struct Box3 {
  double lo[3], hi[3];
};

__global__ void __launch_bounds__(256)
k_mesh_coords(int dim, int n0, int n1, int n2, const __grid_constant__ Box3 bx, long long nv, double* __restrict__ out) {
  const long long nn0 = n0 + 1, nn1 = dim >= 2 ? n1 + 1 : 1;
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += (long long)gridDim.x * blockDim.x) {
    const long long ix = v % nn0, iy = (v / nn0) % nn1, iz = v / (nn0 * nn1);
    const long long ii[3] = {ix, iy, iz};
    const int n[3] = {n0, n1, n2};
    for (int k = 0; k < dim; ++k) {
      const double a = bx.lo[k], b = bx.hi[k];
      double xk;
      if (dim == 3)  // BoxMesh: a + (i*(b-a))/n
        xk = __dadd_rn(a, __ddiv_rn(__dmul_rn((double)ii[k], __dsub_rn(b, a)), (double)n[k]));
      else           // IntervalMesh / RectangleMesh: a + ((b-a)/n)*i
        xk = __dadd_rn(a, __dmul_rn(__ddiv_rn(__dsub_rn(b, a), (double)n[k]), (double)ii[k]));
      out[v * dim + k] = xk;
    }
  }
}

int launch_mesh_coords_box(pde_ctx* c, int dim, const int32_t n[3], const double lo[3], const double hi[3], double* out) {
  int64_t nv, ncell;
  PDE_OK(pde_mesh_counts(dim, n, &nv, &ncell));
  Box3 bx;
  for (int k = 0; k < 3; ++k) { bx.lo[k] = k < dim ? lo[k] : 0.0; bx.hi[k] = k < dim ? hi[k] : 0.0; }
  int blocks = flat_blocks(c, nv, 256);
  k_mesh_coords<<<blocks, 256, 0, c->stream>>>(dim, n[0], dim > 1 ? n[1] : 0, dim > 2 ? n[2] : 0, bx, nv, out);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int launch_mesh_coords(pde_ctx* c, int dim, const int32_t n[3], const double L[3], double* out) {
  const double lo[3] = {0.0, 0.0, 0.0};
  return launch_mesh_coords_box(c, dim, n, lo, L, out);
}

__device__ __forceinline__ void sort_small(long long* v, int n) {
  for (int i = 1; i < n; ++i) {
    long long key = v[i];
    int j = i - 1;
    while (j >= 0 && v[j] > key) { v[j + 1] = v[j]; --j; }
    v[j + 1] = key;
  }
}

__global__ void __launch_bounds__(256)
k_mesh_cells(int dim, int n0, int n1, int n2, long long ngrid, int sorted, int ncomp, int layout, long long nv,
             int32_t* __restrict__ out) {
  const int tets[6][4] = {{0, 1, 3, 7}, {0, 1, 7, 5}, {0, 5, 7, 4}, {0, 3, 2, 7}, {0, 6, 4, 7}, {0, 2, 6, 7}};
  const int tris[2][3] = {{0, 1, 3}, {0, 2, 3}};
  const int nsimp = dim == 1 ? 1 : (dim == 2 ? 2 : 6);
  const int nvs = dim + 1;
  const long long nn0 = n0 + 1, nn1 = n1 + 1;
  for (long long gcell = (long long)blockIdx.x * blockDim.x + threadIdx.x; gcell < ngrid;
       gcell += (long long)gridDim.x * blockDim.x) {
    long long ix = gcell % n0, iy = 0, iz = 0;
    if (dim >= 2) iy = (gcell / n0) % n1;
    if (dim == 3) iz = gcell / ((long long)n0 * n1);
    long long v[8];
    v[0] = dim == 1 ? ix : (dim == 2 ? iy * nn0 + ix : iz * nn0 * nn1 + iy * nn0 + ix);
    v[1] = v[0] + 1;
    v[2] = v[0] + nn0;
    v[3] = v[1] + nn0;
    for (int q = 0; q < 4; ++q) v[4 + q] = v[q] + nn0 * nn1;
    for (int t = 0; t < nsimp; ++t) {
      long long s[4];
      for (int a = 0; a < nvs; ++a) s[a] = v[dim == 1 ? a : (dim == 2 ? tris[t][a] : tets[t][a])];
      if (sorted) sort_small(s, nvs);
      int32_t* dst = out + (gcell * nsimp + t) * (long long)(nvs * ncomp);
      for (int cc = 0; cc < ncomp; ++cc)
        for (int a = 0; a < nvs; ++a)
          dst[cc * nvs + a] = (int32_t)(ncomp == 1 ? s[a] : (layout == 0 ? cc * nv + s[a] : ncomp * s[a] + cc));
    }
  }
}

int launch_mesh_cells(pde_ctx* c, int dim, const int32_t n[3], int sorted, int ncomp, int layout, int32_t* out) {
  int64_t nv, ncell;
  PDE_OK(pde_mesh_counts(dim, n, &nv, &ncell));
  long long ngrid = ncell / (dim == 1 ? 1 : (dim == 2 ? 2 : 6));
  int blocks = flat_blocks(c, ngrid, 256);
  k_mesh_cells<<<blocks, 256, 0, c->stream>>>(dim, n[0], dim > 1 ? n[1] : 1, dim > 2 ? n[2] : 1, ngrid, sorted, ncomp,
                                               layout, nv, out);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

__global__ void __launch_bounds__(128)
k_bc_mask(const __grid_constant__ Grid g, const __grid_constant__ BcDev bc, uint8_t* __restrict__ mask,
          double* __restrict__ vals) {
  const long long rows = (long long)g.nn[1] * g.nzl;
  for (long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y; row < rows;
       row += (long long)gridDim.x * blockDim.y) {
    const int iy = (int)(row % g.nn[1]);
    const int lz = (int)(row / g.nn[1]);
    for (int ix = threadIdx.x; ix < g.nn[0]; ix += blockDim.x) {
      double bcv = 0.0;
      const bool isdir = bc_node(g, bc, ix, iy, lz + g.z0, &bcv);
      const long long node = row * g.nn[0] + ix;
      mask[node] = isdir ? 1 : 0;
      if (vals) vals[node] = isdir ? bcv : 0.0;
    }
  }
}

int launch_bc_mask(pde_ctx* c, const Grid& g, const BcDev& bc, uint8_t* mask, double* vals) {
  RowLaunch rl = row_launch(c, g);
  k_bc_mask<<<rl.grid, rl.block, 0, c->stream>>>(g, bc, mask, vals);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
