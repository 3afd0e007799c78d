// k_elast3d: the 3-D P1 elasticity operator (reference forms fenics_mcp_server.py:1808-1828) as a TMA-fed plane
// sweep with every tile transfer done by the TMA unit, for sm_100a.
//
// What differs from the generic vector instantiation k_sweep3d<3, ...> (stencil3d.cu), which it replaces on the hot path:
//   * the 15 3x3 blocks of the Kuhn-mesh operator are never touched as 111 coefficients.  On a uniform Kuhn mesh
//       K^{aa} = 7-point stencil (centre, +-x, +-y, +-z)                                 12 numbers
//       K^{ab} = u_ab * fixed integer pattern, a != b (u_xy ~ hz, u_xz ~ hy, u_yz ~ hx)   3 numbers
//     (SURVEY A.2/A.6: all couplings are (lambda+mu) x a pure-geometry stencil), so the whole operator is 15 doubles that
//     live in uniform registers, and the integer patterns are folded into shared differences: 83 FP64 operations per
//     node instead of 120, no LDC/R2UR coefficient traffic.  The host checks the table against the pattern and
//     falls back to the generic kernel if it does not match.
//   * tile geometry is a compile-time constant (32 x 8 nodes, 128 threads, thread = one column x two rows), so every
//     shared-memory access is base + immediate.
//   * the right-hand side / previous iterate of the retiring plane arrive by TMA in the same pipeline stage as the input
//     plane; every thread stores its own outputs (a TMA-store epilogue through shared memory measured the same on B200).
//   * the input components are processed one after the other into the nine accumulators of a row, which keeps the
//     kernel at <= 128 registers: four CTAs (16 warps) per SM instead of two.
// Rows with an incomplete element patch (natural faces) are left to k_face_rows, exactly as in k_sweep3d: this kernel
// does not store them.
#include <cuda.h>

#include <cmath>

#include <type_traits>

#include "device.cuh"
#include "tma.cuh"

namespace {

// tile width / strips per tile / pipeline depth: compile-time so that every shared-memory access is base + immediate
// (A/B builds: PDE_B200_NVCC_FLAGS="-DE_TX_=64 -DE_NS_=4")
#ifndef E_TX_
#define E_TX_ 32
#endif
#ifndef E_NS_
#define E_NS_ 4
#endif
#ifndef E_STAGES_
#define E_STAGES_ 4
#endif
constexpr int E_TX = E_TX_, E_NS = E_NS_;          // a warp owns (part of) one strip of YS rows across the tile
constexpr int E_BX = E_TX + 4;                     // input box: origin (x0-2, y0-1) (the TMA start must be 16-byte aligned)
constexpr int E_STAGES = E_STAGES_;
static_assert(E_TX % 32 == 0, "strips must not share a warp");
constexpr int E_NT = E_TX * E_NS;
struct EG {
  static constexpr int YS = 2;                     // rows per strip
  static constexpr int TY = E_NS * YS;             // rows per tile
  static constexpr int BY = TY + 2;
  static constexpr int XCOMP = E_BX * BY;          // doubles per component of an input box
  static constexpr int XBOX = 3 * XCOMP;           // doubles that arrive per input box
  static constexpr int XSTAGE = (XBOX + 15) / 16 * 16;   // padded: every TMA destination stays 128-byte aligned
  static constexpr int TCOMP = E_TX * TY;
  static constexpr int TILE = 3 * TCOMP;           // one plane of the output tile, three components
  static_assert((TILE * 8) % 128 == 0, "TMA destinations must stay 128-byte aligned");
};

enum { EM_APPLY = 0, EM_RESID = 1, EM_CHEBY = 2, EM_FIRST2 = 3 };

struct ECoef {
  double k0[3], kx[3], ky[3], kz[3];   // K^{aa}: centre, +-x, +-y, +-z
  // coupling units, indexed by the INPUT component B they multiply (all equal in B for the plain operator; the fused
  // first-two-sweeps mode folds the column scaling s0 / diag[B] of x1 = s0 D^-1 b into them); uxy2 = 2 uxy
  double uxy[3], uxz[3], uyz[3], uxy2[3];
};
struct EArgs {
  double* y;
  double bB[3];    // apply: bscale * bconst[c] * load
  double c2d[3];   // Chebyshev: c2 / diag[c]
  double ascale, bscale, c1;
  int prev_mode, do_reduce, has_y, need_yy;
};
struct EGeom {
  int nn0, nn1, nzl, z0, nzg;
  int ntx, nty, nzc, zc;
  int on[6], side_excl;
  int PX;
  long long plane, comp_stride;
};

// Contribution of input component B of the resident plane to the outputs one plane below (aP: this plane is their
// dz=+1 neighbour), in the plane (a0) and one plane above (aM: dz=-1; started here when B == 0).
//   V[r][c]: plane values at strip rows r-1 (r = 0..YS+1), columns c-1 (c = 0..2); V[0][2] and V[YS+1][0] are unused.
// Coupling patterns in units u_ab (offsets 0, +-x, +-y, +-z, +-(x+y), +-(x+z), +-(y+z), +-(x+y+z)):
//   xy: -4  2  2 -1 -2  1  1 -1      xz: -4  2 -1  2  1 -2  1 -1      yz: -4 -1  2  2  1  1 -2 -1
template <int B, int YS>
__device__ __forceinline__ void e_contrib(const ECoef& C, const double (&V)[YS + 2][3], double (&aP)[YS][3],
                                          double (&a0)[YS][3], double (&aM)[YS][3]) {
  double P[YS + 2], Q[YS + 2];
  if (B != 1) {
#pragma unroll
    for (int r = 1; r <= YS + 1; ++r) P[r] = V[r][1] - V[r][2];
#pragma unroll
    for (int r = 0; r <= YS; ++r) Q[r] = V[r][1] - V[r][0];
  }
#pragma unroll
  for (int j = 0; j < YS; ++j) {
    const int r = j + 1;
    const double f0 = V[r][1];
    const double Sx = V[r][2] + V[r][0];
    const double Sy = V[r + 1][1] + V[r - 1][1];
    const double Sd = V[r + 1][2] + V[r - 1][0];
    a0[j][B] = fma(C.k0[B], f0, fma(C.kx[B], Sx, fma(C.ky[B], Sy, a0[j][B])));
    const double M = fma(-2.0, f0, (Sx + Sy) - Sd);           // xy pattern / 2
    if (B == 0) {
      a0[j][1] = fma(C.uxy2[B], M, a0[j][1]);
      a0[j][2] = fma(C.uxz[B], fma(3.0, fma(-2.0, f0, Sx), -M), a0[j][2]);
    } else if (B == 1) {
      a0[j][0] = fma(C.uxy2[B], M, a0[j][0]);
      a0[j][2] = fma(C.uyz[B], fma(3.0, fma(-2.0, f0, Sy), -M), a0[j][2]);
    } else {
      a0[j][0] = fma(C.uxz[B], fma(3.0, fma(-2.0, f0, Sx), -M), a0[j][0]);
      a0[j][1] = fma(C.uyz[B], fma(3.0, fma(-2.0, f0, Sy), -M), a0[j][1]);
    }
    // dz = +1: g0 = V[r][1], gx = V[r][2], gy = V[r+1][1], gd = V[r+1][2]
    aP[j][B] = fma(C.kz[B], f0, aP[j][B]);
    if (B == 0) {
      aP[j][1] = fma(C.uxy[B], P[r + 1] - P[r], aP[j][1]);
      aP[j][2] = fma(C.uxz[B], fma(2.0, P[r], P[r + 1]), aP[j][2]);
    } else if (B == 1) {
      const double R1 = V[r][1] - V[r + 1][1], R2 = V[r][2] - V[r + 1][2];
      aP[j][0] = fma(C.uxy[B], R2 - R1, aP[j][0]);
      aP[j][2] = fma(C.uyz[B], fma(2.0, R1, R2), aP[j][2]);
    } else {
      const double Exz = fma(2.0, P[r], P[r + 1]);
      aP[j][0] = fma(C.uxz[B], Exz, aP[j][0]);
      aP[j][1] = fma(C.uyz[B], fma(3.0, V[r][2] - V[r + 1][1], Exz), aP[j][1]);
    }
    // dz = -1: g0 = V[r][1], gx = V[r][0], gy = V[r-1][1], gd = V[r-1][0]
    if (B == 0) {
      aM[j][0] = C.kz[0] * f0;
      aM[j][1] = C.uxy[B] * (Q[r - 1] - Q[r]);
      aM[j][2] = C.uxz[B] * fma(2.0, Q[r], Q[r - 1]);
    } else if (B == 1) {
      const double R1 = V[r][1] - V[r - 1][1], R2 = V[r][0] - V[r - 1][0];
      aM[j][1] = fma(C.kz[1], f0, aM[j][1]);
      aM[j][0] = fma(C.uxy[B], R2 - R1, aM[j][0]);
      aM[j][2] = fma(C.uyz[B], fma(2.0, R1, R2), aM[j][2]);
    } else {
      const double Exz = fma(2.0, Q[r], Q[r - 1]);
      aM[j][2] = fma(C.kz[2], f0, aM[j][2]);
      aM[j][0] = fma(C.uxz[B], Exz, aM[j][0]);
      aM[j][1] = fma(C.uyz[B], fma(3.0, V[r][0] - V[r - 1][1], Exz), aM[j][1]);
    }
  }
}

// MODE: EM_APPLY  y = m (ascale A x + bB)            reductions x.y, y.y
//       EM_RESID  y = m (ascale A x + bscale b)       reductions x.y, y.y
//       EM_CHEBY  y = x + m (c1 d + c2 D^-1 (b - A x)) reduction b.y ; d = x - x_prev (PREV: x_prev is loaded),
//                 x (prev_mode 2: the previous iterate is zero) or 0 (restart)
//       EM_FIRST2 the first TWO sweeps from a zero guess in one pass: the input field is the right-hand side b, the
//                 coefficients arrive with their columns scaled by s0 / diag (so the stencil yields A x1, x1 = s0 D^-1 b),
//                 y = (1 + c1) x1 + c2 D^-1 (b - A x1).  Valid where every neighbour carries the interior diagonal:
//                 rows on AND next to natural faces are left to k_face_rows (two layers), which knows the class diagonals
#ifndef E_THREADS_PER_SM
#define E_THREADS_PER_SM 512
#endif
template <int MODE, bool PREV>
__global__ void __launch_bounds__(E_NT, E_THREADS_PER_SM / E_NT)
k_elast3d(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmb,
          const __grid_constant__ CUtensorMap tmp, const __grid_constant__ ECoef C, const __grid_constant__ EArgs a,
          const __grid_constant__ EGeom ge, ReduceBuf red, double* red_out, const double* face_part, int nface_part) {
  using G = EG;
  constexpr int YS = G::YS;
  constexpr bool HAS_B = MODE == EM_RESID || MODE == EM_CHEBY;
  constexpr bool CHEBY = MODE == EM_CHEBY;
  constexpr bool FIRST2 = MODE == EM_FIRST2;
  constexpr int NAUX = (HAS_B ? 1 : 0) + (PREV ? 1 : 0);
  constexpr int STAGE_ELEMS = G::XSTAGE + NAUX * G::TILE;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* const stage0 = reinterpret_cast<double*>(smem_raw);
  uint64_t* const bars = reinterpret_cast<uint64_t*>(stage0 + E_STAGES * STAGE_ELEMS);

  const int t = threadIdx.x;
  const int item = blockIdx.x;
  const int itx = item % ge.ntx;
  const int ity = (item / ge.ntx) % ge.nty;
  const int izc = item / (ge.ntx * ge.nty);
  const int x0 = itx * E_TX, y0 = ity * G::TY;
  const int za = izc * ge.zc;
  const int zb = min(za + ge.zc, ge.nzl);
  const int nplanes = zb - za + 2;   // input planes za-1 .. zb
  const uint32_t bar0 = smem_u32(bars);
  const uint32_t stg0 = smem_u32(stage0);
  constexpr uint32_t STAGE_BYTES = STAGE_ELEMS * 8;

  // step n: input plane za-1+n, and (n >= 2) the right-hand side / previous iterate of output plane za+n-2
  auto issue = [&](int n) {
    const uint32_t bar = bar0 + 8 * (n % E_STAGES);
    const uint32_t dst = stg0 + (n % E_STAGES) * STAGE_BYTES;
    const bool aux = NAUX > 0 && n >= 2;
    mbar_expect_tx(bar, (uint32_t)(G::XBOX * 8 + (aux ? NAUX * G::TILE * 8 : 0)));
    tma_load_4d(dst, &tmx, x0 - 2, y0 - 1, za - 1 + n + PDE_NG, 0, bar);
    if (aux) {
      if (HAS_B) tma_load_4d(dst + G::XSTAGE * 8, &tmb, x0, y0, za + n - 2 + PDE_NG, 0, bar);
      if (PREV) tma_load_4d(dst + (G::XSTAGE + G::TILE) * 8, &tmp, x0, y0, za + n - 2 + PDE_NG, 0, bar);
    }
  };
  if (t == 0) {
#pragma unroll
    for (int s = 0; s < E_STAGES; ++s) mbar_init(bar0 + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (t == 0)
    for (int n = 0; n < E_STAGES - 1 && n < nplanes; ++n) issue(n);

  const int lx = t % E_TX;
  const int st = t / E_TX;
  const int ix = x0 + lx;
  const int iy0 = y0 + st * YS;
  const int xoff = (st * YS) * E_BX + lx + 1;   // V[r][c] of component q: stage[q*XCOMP + xoff + r*E_BX + c]
  const int toff = (st * YS) * E_TX + lx;       // tile element (q, row j): [q*TCOMP + toff + j*E_TX]

  // row flags (bit j = row j of the strip), constant over the march.  fre: inside the domain and not Dirichlet through
  // an x/y face; slow: free but on a natural x/y face (k_face_rows computes it); okb: inside the domain.
  unsigned fre = 0, slow = 0, okb = 0;
  bool z_excl = false;   // "other_faces" rule of the reference: the z faces skip the x-end columns
  {
    const bool xin = ix < ge.nn0;
    const bool xe0 = ix == 0, xe1 = ix == ge.nn0 - 1;
    z_excl = ge.side_excl && (xe0 || xe1);
#pragma unroll
    for (int j = 0; j < YS; ++j) {
      const int iy = iy0 + j;
      const bool ye0 = iy == 0, ye1 = iy == ge.nn1 - 1;
      bool d = (xe0 && ge.on[0]) || (xe1 && ge.on[1]);
      if (!d && !z_excl) d = (ye0 && ge.on[2]) || (ye1 && ge.on[3]);
      const bool in = xin && iy < ge.nn1;
      if (in) okb |= 1u << j;
      if (in && !d) fre |= 1u << j;
      bool sl = xe0 || xe1 || ye0 || ye1;
      // fused first sweeps: also the layer next to a NATURAL x / y face (its neighbours carry another diagonal)
      if (FIRST2) sl = sl || (ix == 1 && !ge.on[0]) || (ix == ge.nn0 - 2 && !ge.on[1]) || (iy == 1 && !ge.on[2]) ||
                       (iy == ge.nn1 - 2 && !ge.on[3]);
      if (in && !d && sl) slow |= 1u << j;
    }
  }
  const unsigned fast = fre & ~slow;            // rows this kernel computes on a generic plane
  double* yrun = a.y + ((long long)ge.PX * iy0 + ix) + ge.plane * za;   // output column at plane za

  double accA[YS][3], accB[YS][3], accC[YS][3];
#pragma unroll
  for (int j = 0; j < YS; ++j)
#pragma unroll
    for (int q = 0; q < 3; ++q) accA[j][q] = accB[j][q] = accC[j][q] = 0.0;
  double red_xy = 0.0, red_yy = 0.0;

  // One pipeline step: input plane za-1+i is resident in stage i % STAGES; output plane za+i-2 retires (FIN).
  auto body = [&](auto fin_tag, int i, double (&aP)[YS][3], double (&a0)[YS][3], double (&aM)[YS][3]) {
    constexpr bool FIN = decltype(fin_tag)::value;
    const int stage = i % E_STAGES;
    mbar_wait(bar0 + 8 * stage, (uint32_t)((i / E_STAGES) & 1));
    const double* const sx = stage0 + stage * STAGE_ELEMS;
    {
      const double* const sp = sx + xoff;
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        double V[YS + 2][3];
#pragma unroll
        for (int r = 0; r < YS + 2; ++r)
#pragma unroll
          for (int c = 0; c < 3; ++c)
            V[r][c] = ((r == 0 && c == 2) || (r == YS + 1 && c == 0)) ? 0.0 : sp[q * G::XCOMP + r * E_BX + c];
#ifdef E_NOMATH   // memory-only probe build: same transfers and shared-memory reads, (almost) no arithmetic
#pragma unroll
        for (int j = 0; j < YS; ++j) {
          double s = 0.0;
#pragma unroll
          for (int r = 0; r < YS + 2; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c) s += V[r][c];
          aP[j][q] += s; aM[j][q] = s; a0[j][q] += C.k0[q] * s;
        }
#else
        if (q == 0) e_contrib<0, YS>(C, V, aP, a0, aM);
        if (q == 1) e_contrib<1, YS>(C, V, aP, a0, aM);
        if (q == 2) e_contrib<2, YS>(C, V, aP, a0, aM);
#endif
      }
    }
    const int zout = za + i - 2;
    if (FIN) {
      // plane type: generic / Dirichlet (or beyond the domain) / natural z face
      const int gz = zout + ge.z0;
      const bool zface = gz == 0 || gz == ge.nzg - 1 ||
                         (FIRST2 && ((gz == 1 && !ge.on[4]) || (gz == ge.nzg - 2 && !ge.on[5])));
      const bool zface_dir = (gz == 0 && ge.on[4]) || (gz == ge.nzg - 1 && ge.on[5]);
      const bool zdir = gz < 0 || gz > ge.nzg - 1 || (zface_dir && !z_excl);
      const unsigned comp = (zdir || zface) ? 0u : fast;             // rows computed here
      const unsigned keep = zdir ? 0u : (zface ? fre : slow);        // rows left to k_face_rows
      // own-column values of the retiring plane: still resident in the stage of the step before
      const double* const xo_s = stage0 + ((i - 1) % E_STAGES) * STAGE_ELEMS + xoff + E_BX + 1;
      const double* const bt = sx + G::XSTAGE + toff;
      const double* const pt = bt + G::TILE;
      const unsigned stmask = a.has_y ? (okb & ~keep) : 0u;          // rows written by this kernel
#pragma unroll
      for (int j = 0; j < YS; ++j) {
        const bool m = (comp >> j) & 1u;
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const double xo = xo_s[q * G::XCOMP + j * E_BX];
          const double A = aP[j][q];
          double yv;
          if (CHEBY) {
            const double Bv = bt[q * G::TCOMP + j * E_TX];
            double dprev;
            if (PREV) dprev = xo - pt[q * G::TCOMP + j * E_TX];
            else dprev = a.prev_mode == 2 ? xo : 0.0;
            const double dn = m ? fma(a.c1, dprev, a.c2d[q] * (Bv - A)) : 0.0;
            yv = xo + dn;
            red_xy = fma(m ? Bv : 0.0, yv, red_xy);
          } else if (FIRST2) {
            // xo is the right-hand side here; A = A x1 (scaled coefficients)
            yv = m ? fma(a.bB[q], xo, a.c2d[q] * (xo - A)) : 0.0;      // bB = (1 + c1) s0 / diag
          } else {
            const double Bt = HAS_B ? a.bscale * bt[q * G::TCOMP + j * E_TX] : a.bB[q];
            yv = m ? fma(a.ascale, A, Bt) : 0.0;
            red_xy = fma(xo, yv, red_xy);
            if (a.need_yy) red_yy = fma(yv, yv, red_yy);
          }
          if ((stmask >> j) & 1u) yrun[q * ge.comp_stride + j * (long long)ge.PX] = yv;
        }
      }
      yrun += ge.plane;
    }
    __syncthreads();   // stage (i-1) and the tiles of stage i are consumed
    if (t == 0 && i + E_STAGES - 1 < nplanes) issue(i + E_STAGES - 1);
  };

  using T_ = std::true_type;
  using F_ = std::false_type;
  body(F_{}, 0, accA, accB, accC);
  body(F_{}, 1, accB, accC, accA);
  for (int i = 2; i < nplanes; i += 3) {
    body(T_{}, i, accC, accA, accB);
    if (i + 1 < nplanes) body(T_{}, i + 1, accA, accB, accC);
    if (i + 2 < nplanes) body(T_{}, i + 2, accB, accC, accA);
  }

  if (a.do_reduce) {
    if (CHEBY) {
      double v[1] = {red_xy};
      block_reduce_finalize<1>(v, red, red_out, face_part, nface_part);
    } else {
      double v[2] = {red_xy, red_yy};
      block_reduce_finalize<2>(v, red, red_out, face_part, nface_part);
    }
  }
}

// The 15 numbers of the operator, checked against the full interior table (15 offsets x 3x3).
bool extract_coef(const OpDev& op, ECoef* C) {
  const double* h = op.h_int;
  auto H = [&](int k, int i, int j) { return h[k * 9 + i * 3 + j]; };
  double mx = 0;
  for (int q = 0; q < PDE_NOFF * 9; ++q) mx = fmax(mx, fabs(h[q]));
  if (!(mx > 0)) return false;
  for (int c = 0; c < 3; ++c) { C->k0[c] = H(0, c, c); C->kx[c] = H(1, c, c); C->ky[c] = H(3, c, c); C->kz[c] = H(5, c, c); }
  for (int c = 0; c < 3; ++c) {
    C->uxy[c] = -H(13, 0, 1);
    C->uxz[c] = -H(13, 0, 2);
    C->uyz[c] = -H(13, 1, 2);
    C->uxy2[c] = 2.0 * C->uxy[c];
  }
  // offsets: 0 centre, 1/2 +-x, 3/4 +-y, 5/6 +-z, 7/8 +-(x+y), 9/10 +-(x+z), 11/12 +-(y+z), 13/14 +-(x+y+z)
  static const int pat[3][8] = {{-4, 2, 2, -1, -2, 1, 1, -1}, {-4, 2, -1, 2, 1, -2, 1, -1}, {-4, -1, 2, 2, 1, 1, -2, -1}};
  const int pa[3] = {0, 0, 1}, pb[3] = {1, 2, 2};
  const double un[3] = {C->uxy[0], C->uxz[0], C->uyz[0]};
  const double tol = 1e-12 * mx;
  for (int k = 0; k < PDE_NOFF; ++k) {
    const int grp = k == 0 ? 0 : (k + 1) / 2;
    for (int p = 0; p < 3; ++p) {
      const double want = pat[p][grp] * un[p];
      if (fabs(H(k, pa[p], pb[p]) - want) > tol || fabs(H(k, pb[p], pa[p]) - want) > tol) return false;
    }
    for (int c = 0; c < 3; ++c) {
      const double want = k == 0 ? C->k0[c] : (grp == 1 ? C->kx[c] : (grp == 2 ? C->ky[c] : (grp == 3 ? C->kz[c] : 0.0)));
      if (fabs(H(k, c, c) - want) > tol) return false;
    }
  }
  return true;
}

template <int MODE, bool PREV>
int launch_t(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a, const ECoef& C) {
  using G = EG;
  constexpr int NAUX = ((MODE == EM_RESID || MODE == EM_CHEBY) ? 1 : 0) + (PREV ? 1 : 0);
  EGeom ge;
  ge.nn0 = g.nn[0]; ge.nn1 = g.nn[1]; ge.nzl = g.nzl; ge.z0 = g.z0; ge.nzg = g.nzg;
  for (int i = 0; i < 6; ++i) ge.on[i] = bc.on[i];
  ge.side_excl = bc.side_excl;
  ge.PX = g.PX; ge.plane = g.plane; ge.comp_stride = g.comp_stride;
  ge.ntx = (g.nn[0] + E_TX - 1) / E_TX;
  ge.nty = (g.nn[1] + G::TY - 1) / G::TY;
  int zc = 64;
  while (zc > 4 && (long long)ge.ntx * ge.nty * ((g.nzl + zc - 1) / zc) < 8LL * c->sm_count) zc /= 2;
  ge.nzc = (g.nzl + zc - 1) / zc;
  ge.zc = (g.nzl + ge.nzc - 1) / ge.nzc;
  ge.nzc = (g.nzl + ge.zc - 1) / ge.zc;
  const long long items = (long long)ge.ntx * ge.nty * ge.nzc;
  if (items > RED_MAX_BLOCKS) PDE_FAIL("elasticity sweep grid exceeds the reduction buffer");
  const size_t smem = (size_t)E_STAGES * (G::XSTAGE + NAUX * G::TILE) * sizeof(double) + E_STAGES * sizeof(uint64_t);
  auto kern = k_elast3d<MODE, PREV>;
  static bool attr_set = false;
  if (!attr_set) {
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    attr_set = true;
  }
  CUtensorMap tmx, tmb, tmp;
  PDE_OK(field_tensor_map(a.x, g, 3, E_BX, G::BY, &tmx));
  tmb = tmp = tmx;   // unused maps still have to be valid kernel parameters
  if (MODE == EM_RESID || MODE == EM_CHEBY) PDE_OK(field_tensor_map(a.b, g, 3, E_TX, G::TY, &tmb));
  if (PREV) PDE_OK(field_tensor_map(a.xprev, g, 3, E_TX, G::TY, &tmp));
  EArgs ea;
  ea.y = a.y;
  ECoef Cs = C;
  for (int i = 0; i < 3; ++i) {
    ea.bB[i] = a.bscale * a.bconst[i] * op.h_load_int;
    ea.c2d[i] = a.c2 * op.h_dinv_int[i];
    if (MODE == EM_FIRST2) {
      // x1 = s0 D^-1 b: fold the column scaling into the coefficients, y = (1 + c1) x1 + c2 D^-1 (b - A x1)
      const double sg = a.s0 * op.h_dinv_int[i];
      ea.bB[i] = (1.0 + a.c1) * sg;
      Cs.k0[i] *= sg; Cs.kx[i] *= sg; Cs.ky[i] *= sg; Cs.kz[i] *= sg;
      Cs.uxy[i] *= sg; Cs.uxz[i] *= sg; Cs.uyz[i] *= sg; Cs.uxy2[i] *= sg;
    }
  }
  ea.ascale = a.ascale; ea.bscale = a.bscale; ea.c1 = a.c1;
  ea.prev_mode = a.prev_mode;
  ea.do_reduce = a.reduce_slot_xy >= 0;
  ea.has_y = a.y != nullptr;
  ea.need_yy = ea.do_reduce && !a.skip_yy;
  double* out = ea.do_reduce ? c->scal + a.reduce_slot_xy : nullptr;
  // Natural faces.  This kernel never stores the rows of k_face_rows, so that kernel can run FIRST and leave its
  // block sums for this kernel's finalize (no fence + atomic ticket in each of its ~5000 latency-bound blocks).
  int nfp = 0;
  if (!op.uniform_diag) PDE_OK(launch_face_rows(c, g, bc, op, a, &nfp));
  kern<<<(unsigned)items, E_NT, smem, c->stream>>>(tmx, tmb, tmp, Cs, ea, ge, c->red, out, c->face_partials, nfp);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace

// Claims the launch when the operator is the 3-D three-component Kuhn-mesh elasticity operator and the mode is one
// the kernel implements; otherwise *handled stays false and the generic vector sweep runs.
int launch_elast3d(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a, bool* handled) {
  *handled = false;
  if (op.ncomp != 3 || g.dim != 3 || g.nk != PDE_NOFF) return 0;
  if (a.ghost_out || (a.cheby == 1 && (a.prev_mode == 3 || !a.b))) return 0;
  if (a.cheby == 2 && (bc.side_excl || a.reduce_slot_xy >= 0)) return 0;
  if (a.cheby && a.prev_mode == 1 && !a.xprev) return 0;
  ECoef C;
  if (!extract_coef(op, &C)) return 0;
  *handled = true;
  if (a.cheby == 2) return launch_t<EM_FIRST2, false>(c, g, bc, op, a, C);
  if (a.cheby)
    return a.prev_mode == 1 ? launch_t<EM_CHEBY, true>(c, g, bc, op, a, C) : launch_t<EM_CHEBY, false>(c, g, bc, op, a, C);
  return a.b ? launch_t<EM_RESID, false>(c, g, bc, op, a, C) : launch_t<EM_APPLY, false>(c, g, bc, op, a, C);
}

// can the smoother use the fused first-two-sweeps mode on this level?  (the caller must know before it decides between
// one fused launch and cheby_first + sweep)
bool elast3d_first2_ok(const Grid& g, const BcDev& bc, const OpDev& op) {
  if (op.ncomp != 3 || g.dim != 3 || g.nk != PDE_NOFF || bc.side_excl) return false;
  if (!sweep_applicable(g, 3)) return false;
  ECoef C;
  return extract_coef(op, &C);
}
