// Specialised streaming kernels for the 3D hot paths (heat / mass 15-point, elasticity 3x3-block).
// launch_stencil_fast() claims a launch when a specialised kernel applies; otherwise the generic
// table kernel in kernels.cu runs.
//
// k_sweep3d: TMA-fed plane sweep.
//   A CTA owns an (x,y) tile of TX x TY nodes and marches over a chunk of z planes.  One elected
//   thread streams each (TX+4) x (TY+2) plane tile (halo included, out-of-domain elements zero-filled
//   by the TMA unit) into a ring of shared-memory stages with cp.async.bulk.tensor, completion on an
//   mbarrier.  The Kuhn 15-point stencil splits by plane into a 4-point part seen from the plane above
//   (dz=-1), a 7-point in-plane part and a 4-point part seen from the plane below (dz=+1), so every
//   plane is read from shared memory ONCE: while plane q is resident each thread adds its contribution
//   to the three outputs q-1, q, q+1 it keeps in registers, then retires output q-1.  A thread owns a
//   strip of YS nodes along y, which cuts shared-memory reads to (3*YS+4)/YS values per output.
//   Algorithmic HBM traffic: read x once, write y once (16 B/dof; Chebyshev sweep 40 B/dof).
//   Nodes whose element patch is incomplete (natural / traction-free faces) are skipped here and computed
//   by k_face_rows (kernels.cu) from the 27-class table right after; Dirichlet rows are masked.
#include <cuda.h>

#include <cmath>

#include <algorithm>
#include <map>
#include <mutex>
#include <type_traits>

#include "device.cuh"
#include "tma.cuh"

#define SW_STAGES 4

struct SweepGeom {
  int tx, ty;         // tile size in nodes
  int bx, by;         // TMA box = (tx+4, ty+2), origin (x0-2, y0-1)
  int ntx, nty, nzc;  // tiles / z-chunks
  int zc;             // planes per chunk
  int ns;             // strips (of YS rows) per tile
  int stage_elems;    // doubles per stage (all components), multiple of 16
  int zlo, zhi;       // output plane range [zlo, zhi): [0, nzl), or [-1, nzl+1) when the ghost planes are computed too
};

template <int NC>
struct Coef {
  double c[PDE_NOFF][NC * NC];
};

struct SweepArgs {
  const double* x;
  const double* b;
  double* y;
  const double* xprev;  // Chebyshev: previous iterate (may alias y); d_{k-1} = x_k - x_{k-1} is never stored
  int prev_mode;        // 0 restart, 1 xprev pointer, 2 previous iterate is zero, 3 previous iterate = s0*dinv*b
  double bconst[3];
  double bscale, ascale, c1, c2, s0;
  double load_int;    // load of the interior class
  double dinv_int[3]; // Jacobi diagonal inverse of the interior class
  int do_reduce;
};

// acc[i] += sum_j C[k][i][j] * v[j].  OFFD: the block has a structurally zero diagonal (elasticity blocks of
// the face- and body-diagonal offsets couple different components only), so those products are skipped.
template <int NC, bool OFFD>
__device__ __forceinline__ void blk_fma(double (&acc)[NC], const Coef<NC>& C, int k, const double (&v)[NC]) {
#pragma unroll
  for (int i = 0; i < NC; ++i)
#pragma unroll
    for (int j = 0; j < NC; ++j)
      if (!(OFFD && i == j)) acc[i] = fma(C.c[k][i * NC + j], v[j], acc[i]);
}
template <int NC, bool OFFD>
__device__ __forceinline__ void blk_set(double (&acc)[NC], const Coef<NC>& C, int k, const double (&v)[NC]) {
#pragma unroll
  for (int i = 0; i < NC; ++i) {
    bool first = true;
    acc[i] = 0.0;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
      if (OFFD && i == j) continue;
      acc[i] = first ? C.c[k][i * NC + j] * v[j] : fma(C.c[k][i * NC + j], v[j], acc[i]);
      first = false;
    }
  }
}

// One resident plane: V[r][c] = plane values at strip rows r-1 (r = 0..YS+1), columns c-1 (c = 0..2).
//   aP (output one plane below) gets the dz=+1 part, a0 the in-plane part, aM (output one plane above)
//   is started with the dz=-1 part.
// Vector operators (NC > 1): the block at -d equals the block at +d (each block is symmetric and the
// operator is symmetric), so the in-plane neighbour pairs are summed before the block product.
template <int NC, int YS>
__device__ __forceinline__ void plane_contrib(const Coef<NC>& C, const double (&V)[YS + 2][3][NC],
                                              double (&aP)[YS][NC], double (&a0)[YS][NC], double (&aM)[YS][NC]) {
  constexpr bool VEC = NC > 1;
#pragma unroll
  for (int j = 0; j < YS; ++j) {
    const int r = j + 1;
    // in-plane: centre, +-x, +-y, +-(x,y)
    blk_fma<NC, false>(a0[j], C, 0, V[r][1]);
    if (VEC) {
      double sx[NC], sy[NC], sd[NC];
#pragma unroll
      for (int q = 0; q < NC; ++q) {
        sx[q] = V[r][2][q] + V[r][0][q];
        sy[q] = V[r + 1][1][q] + V[r - 1][1][q];
        sd[q] = V[r + 1][2][q] + V[r - 1][0][q];
      }
      blk_fma<NC, false>(a0[j], C, 1, sx);
      blk_fma<NC, false>(a0[j], C, 3, sy);
      blk_fma<NC, true>(a0[j], C, 7, sd);
    } else {
      blk_fma<NC, false>(a0[j], C, 1, V[r][2]);
      blk_fma<NC, false>(a0[j], C, 2, V[r][0]);
      blk_fma<NC, false>(a0[j], C, 3, V[r + 1][1]);
      blk_fma<NC, false>(a0[j], C, 4, V[r - 1][1]);
      blk_fma<NC, false>(a0[j], C, 7, V[r + 1][2]);
      blk_fma<NC, false>(a0[j], C, 8, V[r - 1][0]);
    }
    // this plane is dz=+1 for the output below: (0,0,1), (1,0,1), (0,1,1), (1,1,1)
    blk_fma<NC, false>(aP[j], C, 5, V[r][1]);
    blk_fma<NC, VEC>(aP[j], C, 9, V[r][2]);
    blk_fma<NC, VEC>(aP[j], C, 11, V[r + 1][1]);
    blk_fma<NC, VEC>(aP[j], C, 13, V[r + 1][2]);
    // this plane is dz=-1 for the output above: (0,0,-1), (-1,0,-1), (0,-1,-1), (-1,-1,-1)
    blk_set<NC, false>(aM[j], C, 6, V[r][1]);
    blk_fma<NC, VEC>(aM[j], C, 10, V[r][0]);
    blk_fma<NC, VEC>(aM[j], C, 12, V[r - 1][1]);
    blk_fma<NC, VEC>(aM[j], C, 14, V[r - 1][0]);
  }
}

// MODE: 0 apply (B = bconst*load), 1 residual-type (B from field b), 2 Chebyshev sweep, 3 fused first TWO
// Chebyshev sweeps from a zero guess (input field = right-hand side; needs a uniform Jacobi diagonal)
enum { M_APPLY = 0, M_RESID = 1, M_CHEBY = 2, M_FIRST2 = 3 };

// launch bounds, tuned on B200 (A/B builds): scalar kernel 192 threads x >= 3 CTAs/SM (<= 113 registers);
// the vector kernel is better left unconstrained (254 registers, 2 CTAs of 128 threads)
#ifndef SW_MAXT1
#define SW_MAXT1 192
#endif
#ifndef SW_MAXT3
#define SW_MAXT3 256
#endif
#ifndef SW_MINB1
#define SW_MINB1 3
#endif
#ifndef SW_MINB3
#define SW_MINB3 1
#endif
template <int NC, int YS, int MODE>
__global__ void __launch_bounds__(NC == 1 ? SW_MAXT1 : SW_MAXT3, NC == 1 ? SW_MINB1 : SW_MINB3)
k_sweep3d(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ Grid g, const __grid_constant__ BcDev bc,
          const __grid_constant__ Coef<NC> C, const __grid_constant__ SweepArgs a, const __grid_constant__ SweepGeom sw,
          ReduceBuf red, double* red_out) {
  constexpr bool CHEBY = MODE >= M_CHEBY;
  constexpr bool HAS_B = MODE == M_RESID || MODE == M_CHEBY;
  constexpr bool LOAD_D = MODE == M_CHEBY;  // loads x_{k-1} (prev_mode 1) to rebuild the direction
  constexpr bool XQ_REG = NC == 1;  // own-column queue in registers; vector kernels re-read x (L2 hit) instead
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* stage0 = reinterpret_cast<double*>(smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)SW_STAGES * sw.stage_elems * sizeof(double));

  const int t = threadIdx.x;
  const int item = blockIdx.x;
  const int itx = item % sw.ntx;
  const int ity = (item / sw.ntx) % sw.nty;
  const int izc = item / (sw.ntx * sw.nty);
  const int x0 = itx * sw.tx, y0 = ity * sw.ty;
  const int za = sw.zlo + izc * sw.zc;
  const int zb = min(za + sw.zc, sw.zhi);
  const int nplanes = zb - za + 2;  // planes za-1 .. zb
  const uint32_t stage_bytes = (uint32_t)(sw.bx * sw.by * NC * sizeof(double));
  const uint32_t bar0 = smem_u32(bars);
  const uint32_t stg0 = smem_u32(stage0);
  const uint32_t stage_stride = (uint32_t)(sw.stage_elems * sizeof(double));

  // full[s]: TMA transaction barrier of stage s (1 arrival + bytes); thread 0 refills a stage after the CTA barrier
  // that follows its last read
  if (t == 0) {
#pragma unroll
    for (int s = 0; s < SW_STAGES; ++s) mbar_init(bar0 + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (t == 0) {
    for (int i = 0; i < SW_STAGES && i < nplanes; ++i) {
      mbar_expect_tx(bar0 + 8 * i, stage_bytes);
      // tensor z coordinate: local plane lz is z = lz + PDE_NG (the ghost planes come first).  The box starts at x0-2: TMA needs
      // the inner start coordinate 16-byte aligned (even for FP64); x0-1 raises an illegal-instruction fault
      tma_load_4d(stg0 + i * stage_stride, &tmx, x0 - 2, y0 - 1, za + i - 1 + PDE_NG, 0, bar0 + 8 * i);
    }
  }

  const int lx = t % sw.tx;
  int st = t / sw.tx;
  const bool active = st < sw.ns;
  if (!active) st = 0;  // surplus threads of the last warp shadow strip 0 and never store
  const int ix = x0 + lx;
  const int iy0 = y0 + st * YS;
  const int comp_elems = sw.bx * sw.by;
  // smem offset of V[0][0]: box row st*YS (= y -1), box column lx+1 (= x -1)
  const double* sbase = stage0 + (st * YS) * sw.bx + lx + 1;

  // per-thread node flags, constant over the z march: bit j describes node (ix, iy0+j).
  //   mrow[j] = 0 for Dirichlet / out-of-range nodes, 1 for free nodes: masked rows need no branch.
  unsigned valid = 0, slowxy = 0, freexy = 0;  // freexy: valid and not Dirichlet through an x/y face
  double mrow[YS];
  bool z_excl = false;  // "other_faces" predicate: side faces skip the x-end columns
#pragma unroll
  for (int j = 0; j < YS; ++j) mrow[j] = 0.0;
  if (active && ix < g.nn[0]) {
    const bool xe0 = ix == 0, xe1 = ix == g.nn[0] - 1;
    z_excl = bc.side_excl && (xe0 || xe1);
#pragma unroll
    for (int j = 0; j < YS; ++j) {
      const int iy = iy0 + j;
      if (iy >= g.nn[1]) continue;
      valid |= 1u << j;
      const bool ye0 = iy == 0, ye1 = iy == g.nn[1] - 1;
      bool d = (xe0 && bc.on[0]) || (xe1 && bc.on[1]);
      if (!d && !z_excl) d = (ye0 && bc.on[2]) || (ye1 && bc.on[3]);
      mrow[j] = d ? 0.0 : 1.0;
      if (!d) freexy |= 1u << j;
      if (!d && (xe0 || xe1 || ye0 || ye1)) slowxy |= 1u << j;
    }
  }
  const long long col0 = (long long)g.PX * iy0 + ix;  // flat offset of (ix, iy0) inside a plane
  const unsigned col0u = (unsigned)col0;
  // Everything the epilogue needs is static per thread except three plane-uniform cases (generic plane, Dirichlet
  // z face, natural z face): row masks as 0/1 doubles, store masks as bit sets, the output column as a pointer.
  //   generic plane : interior-class rows computed, rows on natural x/y faces left to k_face_rows (not stored)
  //   Dirichlet face: every valid row stores 0
  //   natural z face: every free row belongs to k_face_rows; only the x/y-Dirichlet rows store 0
  double mgen[YS];
#pragma unroll
  for (int j = 0; j < YS; ++j) mgen[j] = ((slowxy >> j) & 1u) ? 0.0 : mrow[j];
  const unsigned st_gen = valid & ~slowxy, st_zface = valid & ~freexy;
  const bool has_y = a.y != nullptr;
  double* const ycol = a.y + col0;   // never dereferenced when a.y is null
  const double* const bcol0 = a.b + col0;       // likewise for a.b / a.xprev
  const double* const dcol0 = a.xprev + col0;
  const double* const xcol0 = a.x + col0;
  const long long pxb = g.PX;

  double accA[YS][NC], accB[YS][NC], accC[YS][NC];
  // own-column values of the resident plane; the plane read one step earlier is the one that retires
  double xA[YS][NC], xB[YS][NC], xC[YS][NC];
#pragma unroll
  for (int j = 0; j < YS; ++j)
#pragma unroll
    for (int i = 0; i < NC; ++i) accA[j][i] = accB[j][i] = accC[j][i] = xA[j][i] = xB[j][i] = xC[j][i] = 0.0;
  double red_xy = 0.0, red_yy = 0.0;

  // One pipeline step: plane q = za-1+i is resident in stage i%STAGES; output plane q-1 retires (FIN).
  auto body = [&](auto fin_tag, int i, double (&aP)[YS][NC], double (&a0)[YS][NC], double (&aM)[YS][NC],
                  double (&xprev)[YS][NC], double (&xcur)[YS][NC]) {
    constexpr bool FIN = decltype(fin_tag)::value;
    const int stage = i % SW_STAGES;
    const uint32_t parity = (uint32_t)((i / SW_STAGES) & 1);
    const int zout = za + i - 2;
    // early global loads for the retiring outputs (consumed after the stencil arithmetic)
    double bv[YS][NC], dv[YS][NC], xv[YS][NC];
    if (FIN && (HAS_B || LOAD_D || !XQ_REG)) {
      // column pointers of this thread at plane zout: one 64-bit add per array and plane, rows and components
      // by running pointers (a full address rebuild per load costs ~6 instructions)
      const long long pofs = (long long)g.plane * zout;
      const bool use_d = LOAD_D && a.prev_mode == 1;
      const double* bcol = HAS_B ? bcol0 + pofs : nullptr;
      const double* dcol = use_d ? dcol0 + pofs : nullptr;
      const double* xcol = xcol0 + pofs;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const double* bp = bcol;
        const double* dp = dcol;
        const double* xp = xcol;
#pragma unroll
        for (int j = 0; j < YS; ++j) {
          const bool ok = (valid >> j) & 1u;
          if (HAS_B) { bv[j][c] = ok ? *bp : 0.0; bp += pxb; }
          if (LOAD_D) { dv[j][c] = (ok && use_d) ? *dp : 0.0; dp += pxb; }   // x_{k-1}
          if (!XQ_REG) { xv[j][c] = ok ? *xp : 0.0; xp += pxb; }
        }
        if (HAS_B) bcol += g.comp_stride;
        if (LOAD_D) dcol += g.comp_stride;
        xcol += g.comp_stride;
      }
    }
    if (FIN && XQ_REG) {
#pragma unroll
      for (int j = 0; j < YS; ++j)
#pragma unroll
        for (int c = 0; c < NC; ++c) xv[j][c] = xprev[j][c];
    }
    mbar_wait(bar0 + 8 * stage, parity);
    {
      double V[YS + 2][3][NC];
      const double* sp = sbase + (size_t)stage * sw.stage_elems;
#pragma unroll
      for (int r = 0; r < YS + 2; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          if ((r == 0 && c == 2) || (r == YS + 1 && c == 0)) {
#pragma unroll
            for (int q = 0; q < NC; ++q) V[r][c][q] = 0.0;  // never used
          } else {
#pragma unroll
            for (int q = 0; q < NC; ++q) V[r][c][q] = sp[q * comp_elems + r * sw.bx + c];
          }
        }
      if (XQ_REG) {
#pragma unroll
        for (int j = 0; j < YS; ++j)
#pragma unroll
          for (int q = 0; q < NC; ++q) xcur[j][q] = V[j + 1][1][q];
      }
      plane_contrib<NC, YS>(C, V, aP, a0, aM);
    }
    __syncthreads();  // every thread has consumed this stage
    if (t == 0 && i + SW_STAGES < nplanes) {
      mbar_expect_tx(bar0 + 8 * stage, stage_bytes);
      tma_load_4d(stg0 + stage * stage_stride, &tmx, x0 - 2, y0 - 1, za + i + SW_STAGES - 1 + PDE_NG, 0, bar0 + 8 * stage);
    }
    if (FIN) {
      const int gz = zout + g.z0;
      const bool ze0 = g.nc[2] > 0 && gz == 0, ze1 = g.nc[2] > 0 && gz == g.nzg - 1;
      const bool zout_dom = gz < 0 || gz > g.nzg - 1;   // ghost plane beyond the domain end: nothing lives there
      const bool zdir = zout_dom || (!z_excl && ((ze0 && bc.on[4]) || (ze1 && bc.on[5])));
      const bool znat = !zdir && (ze0 || ze1);          // natural z face: all free rows go to k_face_rows
      const double mz = (zdir || znat) ? 0.0 : 1.0;
      const unsigned todo = has_y ? (zdir ? valid : (znat ? st_zface : st_gen)) : 0u;   // rows stored by this kernel
      // plane base pointer: one 64-bit add per plane and component, rows by a running pointer
      double* const yplane = ycol + (long long)g.plane * zout;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        double* yp = yplane + c * g.comp_stride;  // may alias xprev: no __restrict__
        const double bB = a.bscale * a.bconst[c] * a.load_int;  // constant load term of the interior class
        const double c2d = a.c2 * a.dinv_int[c];
        const double s0d = a.s0 * a.dinv_int[c];
#pragma unroll
        for (int j = 0; j < YS; ++j) {
          const bool on = (todo >> j) & 1u;
          const double m = mgen[j] * mz;
          if (MODE == M_FIRST2) {
            // zero guess: x1 = d1 = s0 D^-1 b ; r = b - A x1 = b - s0 D^-1 (A b) ; d2 = c1 d1 + c2 D^-1 r
            const double bi = xv[j][c];
            const double d1 = s0d * bi;
            const double dn = m * fma(a.c1, d1, c2d * fma(-s0d, aP[j][c], bi));
            const double yv = m * d1 + dn;
            if (on) *yp = yv;
            red_xy = fma(bi, yv, red_xy);
          } else if (CHEBY) {
            const double B = bv[j][c];
            const double xo = xv[j][c];
            // direction of the previous sweep, rebuilt from the iterates
            const double dprev = a.prev_mode == 1 ? xo - dv[j][c]
                               : (a.prev_mode == 2 ? xo : (a.prev_mode == 3 ? xo - s0d * B : 0.0));
            const double dn = m * fma(a.c1, dprev, c2d * (B - aP[j][c]));
            const double yv = xo + dn;
            if (on) *yp = yv;
            red_xy = fma(m * B, yv, red_xy);
          } else {
            const double yv = m * (HAS_B ? fma(a.ascale, aP[j][c], a.bscale * bv[j][c]) : fma(a.ascale, aP[j][c], bB));
            if (on) *yp = yv;
            red_xy = fma(xv[j][c], yv, red_xy);
            red_yy = fma(yv, yv, red_yy);
          }
          yp += pxb;
        }
      }
    }
  };

  using T_ = std::true_type;
  using F_ = std::false_type;
  // steps 0 and 1 only fill the pipeline; output za retires at step 2
  body(F_{}, 0, accA, accB, accC, xC, xA);
  body(F_{}, 1, accB, accC, accA, xA, xB);
  for (int i = 2; i < nplanes; i += 3) {
    body(T_{}, i, accC, accA, accB, xB, xC);
    if (i + 1 < nplanes) body(T_{}, i + 1, accA, accB, accC, xC, xA);
    if (i + 2 < nplanes) body(T_{}, i + 2, accB, accC, accA, xA, xB);
  }

  if (a.do_reduce) {
    if (CHEBY) {  // sum b.y of a smoother sweep (the preconditioned-CG r.z)
      double v[1] = {red_xy};
      block_reduce_finalize<1>(v, red, red_out);
    } else {
      double v[2] = {red_xy, red_yy};
      block_reduce_finalize<2>(v, red, red_out);
    }
  }
}

// ---- host side: tensor maps, tile geometry, launch ---------------------------------------------------
typedef CUresult (*PFN_tmEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_tmEncodeTiled tm_encode_fn() {
  static PFN_tmEncodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_tmEncodeTiled)p;
  });
  return fn;
}

struct TmKey {
  const void* base;
  int nn0, nn1, nz, nc, bx, by, bz;
  long long px, plane, cs;
  bool operator<(const TmKey& o) const {
    if (base != o.base) return base < o.base;
    if (nn0 != o.nn0) return nn0 < o.nn0;
    if (nn1 != o.nn1) return nn1 < o.nn1;
    if (nz != o.nz) return nz < o.nz;
    if (nc != o.nc) return nc < o.nc;
    if (bx != o.bx) return bx < o.bx;
    if (by != o.by) return by < o.by;
    if (bz != o.bz) return bz < o.bz;
    if (px != o.px) return px < o.px;
    if (plane != o.plane) return plane < o.plane;
    return cs < o.cs;
  }
};

// Tensor map of a padded field: (x, y, z incl. the ghost planes, component); out-of-range x/y -> 0.
int field_tensor_map(const double* field, const Grid& g, int nc, int bx, int by, CUtensorMap* out, int bz) {
  static std::map<TmKey, CUtensorMap> cache;
  static std::mutex mu;
  TmKey k{(const void*)field, g.nn[0], g.nn[1], g.nzl + 2 * PDE_NG, nc, bx, by, bz, g.PX, g.plane, g.comp_stride};
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(k);
  if (it != cache.end()) { *out = it->second; return 0; }
  PFN_tmEncodeTiled enc = tm_encode_fn();
  if (!enc) PDE_FAIL("cuTensorMapEncodeTiled is not available from the CUDA driver");
  cuuint64_t dims[4] = {(cuuint64_t)g.nn[0], (cuuint64_t)g.nn[1], (cuuint64_t)(g.nzl + 2 * PDE_NG), (cuuint64_t)nc};
  cuuint64_t strides[3] = {(cuuint64_t)g.PX * 8, (cuuint64_t)g.plane * 8, (cuuint64_t)g.comp_stride * 8};
  cuuint32_t box[4] = {(cuuint32_t)bx, (cuuint32_t)by, (cuuint32_t)bz, (cuuint32_t)nc};
  cuuint32_t es[4] = {1, 1, 1, 1};
  void* base = (void*)(field - PDE_NG * g.plane);  // first ghost plane below local plane 0
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) PDE_FAIL("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
  if (cache.size() > 8192) cache.clear();
  cache[k] = *out;
  return 0;
}


template <int NC, int YS, int MODE>
static int launch_sweep_t(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a) {
  SweepGeom sw;
  constexpr int maxnt = NC == 1 ? SW_MAXT1 : SW_MAXT3;
  // tile width and threads per CTA tuned on B200 (heat 512^3, elasticity 1280x256x256); two columns of margin for the
  // even rounding of tx (513 nodes: 3 tiles of 172 on 192 threads, A/B: apply 0.397 -> 0.375 ms)
  const int txmax = std::min(NC == 1 ? 192 : 64, maxnt - 2);
  const int nt_target = std::min(NC == 1 ? 192 : 128, maxnt);
  sw.ntx = (g.nn[0] + txmax - 1) / txmax;
  sw.tx = (g.nn[0] + sw.ntx - 1) / sw.ntx;
  sw.tx += sw.tx & 1;  // even: the TMA box row must be a multiple of 16 bytes
  sw.ntx = (g.nn[0] + sw.tx - 1) / sw.tx;
  sw.ns = nt_target / sw.tx;
  if (sw.ns < 1) sw.ns = 1;
  const int max_ns = (g.nn[1] + YS - 1) / YS;
  if (sw.ns > max_ns) sw.ns = max_ns;
  int nt = ((sw.tx * sw.ns + 31) / 32) * 32;
  if (nt > maxnt) PDE_FAIL("sweep tile exceeds the thread limit");
  sw.ty = sw.ns * YS;
  sw.nty = (g.nn[1] + sw.ty - 1) / sw.ty;
  sw.bx = sw.tx + 4;
  sw.by = sw.ty + 2;
  if (sw.bx > 256 || sw.by > 256) PDE_FAIL("sweep TMA box exceeds 256");
  int zc = 64;
  // small grids (coarse multigrid levels): shorter z chunks so that the grid still covers the SMs
  while (zc > 4 && (long long)sw.ntx * sw.nty * ((g.nzl + zc - 1) / zc) < 4LL * c->sm_count) zc /= 2;
  // ghost_out: also produce the two ghost planes next to the slab (needs two valid halo planes of x and one of b),
  // so that the consumer (restriction) needs no halo exchange of the result
  const int gout = (a.ghost_out && op.uniform_diag) ? 1 : 0;
  sw.zlo = -gout;
  sw.zhi = g.nzl + gout;
  const int nzr = sw.zhi - sw.zlo;
  sw.nzc = (nzr + zc - 1) / zc;
  sw.zc = (nzr + sw.nzc - 1) / sw.nzc;
  sw.nzc = (nzr + sw.zc - 1) / sw.zc;
  sw.stage_elems = ((sw.bx * sw.by * NC + 15) / 16) * 16;
  const long long items = (long long)sw.ntx * sw.nty * sw.nzc;
  if (items > RED_MAX_BLOCKS) PDE_FAIL("sweep grid exceeds the reduction buffer");
  const size_t smem = (size_t)SW_STAGES * sw.stage_elems * sizeof(double) + SW_STAGES * sizeof(uint64_t);
  auto kern = k_sweep3d<NC, YS, MODE>;
  static size_t smem_set = 0;
  if (smem > smem_set) {
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  CUtensorMap tm;
  PDE_OK(field_tensor_map(a.x, g, NC, sw.bx, sw.by, &tm));
  Coef<NC> C;
  for (int k = 0; k < PDE_NOFF; ++k)
    for (int q = 0; q < NC * NC; ++q) C.c[k][q] = op.h_int[k * NC * NC + q];
  SweepArgs sa;
  sa.x = a.x; sa.b = a.b; sa.y = a.y; sa.xprev = a.xprev; sa.prev_mode = a.prev_mode;
  for (int i = 0; i < 3; ++i) sa.bconst[i] = a.bconst[i];
  sa.bscale = a.bscale; sa.ascale = a.ascale; sa.c1 = a.c1; sa.c2 = a.c2; sa.s0 = a.s0;
  sa.load_int = op.h_load_int;
  for (int i = 0; i < 3; ++i) sa.dinv_int[i] = i < NC ? op.h_dinv_int[i] : 0.0;
  sa.do_reduce = a.reduce_slot_xy >= 0;
  double* out = sa.do_reduce ? c->scal + a.reduce_slot_xy : nullptr;
  kern<<<(unsigned)items, nt, smem, c->stream>>>(tm, g, bc, C, sa, sw, c->red, out);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  // natural (non-Dirichlet) faces: their rows have incomplete element patches and come from the class table
  if (!op.uniform_diag) PDE_OK(launch_face_rows(c, g, bc, op, a));
  return 0;
}

// does the TMA plane-sweep kernel take this grid?  (callers that rely on its ghost-plane outputs must ask)
bool sweep_applicable(const Grid& g, int ncomp) {
  if (g.dim != 3 || g.nk != PDE_NOFF) return false;
  if (ncomp != 1 && ncomp != 3) return false;
  // small grids (coarse multigrid levels) stay on the generic kernel: they are launch-latency bound
  if (g.nn[0] < 32 || g.nn[1] < 8 || g.nzl < 4) return false;
  if ((long long)g.nn[0] * g.nn[1] * g.nzl < 4096) return false;
  return true;
}

// ----------------------------------------------------------------------------------------------------
// k_sweep2d: the 2-D heat / mass operators (internal axes x and z; rows are contiguous) with every face Dirichlet.
//   A thread owns one column and marches over a chunk of rows keeping the three partial sums of the Kuhn 7-point
//   stencil (centre, +-x, +-z, +-(x,z)) in registers, exactly like the plane march of k_sweep3d: row q contributes
//   to outputs q-1, q and q+1, then output q-1 retires.  Three coalesced loads per row (the +-1 columns hit L1), no
//   shared memory: DRAM sees every element once.  Same modes and epilogues as k_sweep3d<1, ., MODE>.
// ----------------------------------------------------------------------------------------------------
struct Coef2d {
  double c0, cxp, cxm, czp, czm, cdp, cdm;   // offsets (0,0) (+1,0) (-1,0) (0,+1) (0,-1) (+1,+1) (-1,-1)
};

template <int MODE>
__global__ void __launch_bounds__(256)
k_sweep2d(const __grid_constant__ Grid g, const __grid_constant__ Coef2d C, const __grid_constant__ SweepArgs a,
          int zc, int nbx, ReduceBuf red, double* red_out) {
  constexpr bool CHEBY = MODE >= M_CHEBY;
  constexpr bool HAS_B = MODE == M_RESID || MODE == M_CHEBY;
  // 1-D grid (the block reduction indexes its partial sums by blockIdx.x): x block fastest
  const int ix = (int)(blockIdx.x % nbx) * blockDim.x + threadIdx.x;
  const int za = (int)(blockIdx.x / nbx) * zc;
  const int zb = min(za + zc, g.nzl);
  const bool col = ix < g.nn[0];
  const double mx = (col && ix > 0 && ix < g.nn[0] - 1) ? 1.0 : 0.0;
  const long long PX = g.PX;
  // pads and ghost rows are zero (or hold the neighbour slab's rows), so the +-1 columns / rows need no guards;
  // columns beyond the row stay inside the allocation (next row) and are masked
  const double* xc = a.x + ix;                                   // column pointers at row 0
  const double* bc_ = HAS_B ? a.b + ix : nullptr;
  const bool use_d = MODE == M_CHEBY && a.prev_mode == 1;
  const double* dc = use_d ? a.xprev + ix : nullptr;
  double* yc = a.y ? a.y + ix : nullptr;                         // may alias xprev: rows are loaded before they are stored
  const double bB = a.bscale * a.bconst[0] * a.load_int;
  const double c2d = a.c2 * a.dinv_int[0], s0d = a.s0 * a.dinv_int[0];
  double accA = 0.0, accB = 0.0, xprev_own = 0.0;
  double red_xy = 0.0, red_yy = 0.0;
  constexpr int U = 4;   // rows per step: all loads of a step are issued before its arithmetic and stores
  for (int q0 = za - 1; q0 <= zb; q0 += U) {
    double vm[U], v0[U], vp[U], Bv[U], Dv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int q = q0 + u;
      const bool ok = col && q <= zb;
      const double* p = xc + PX * q;
      vm[u] = ok ? p[-1] : 0.0;
      v0[u] = ok ? p[0] : 0.0;
      vp[u] = ok ? p[1] : 0.0;
      const bool rz = ok && q > za;                              // output row z = q-1 retires at this row
      Bv[u] = (HAS_B && rz) ? bc_[PX * (q - 1)] : 0.0;
      Dv[u] = (use_d && rz) ? dc[PX * (q - 1)] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int q = q0 + u;
      if (q > zb) break;
      const double done = fma(C.cdp, vp[u], fma(C.czp, v0[u], accA));          // output row q-1 is complete
      accA = fma(C.cxm, vm[u], fma(C.cxp, vp[u], fma(C.c0, v0[u], accB)));      // row q: in-row part on top of its dz=-1 part
      accB = fma(C.cdm, vm[u], C.czm * v0[u]);                                  // row q+1: dz=-1 part
      if (q > za) {
        const int z = q - 1;
        const int gz = z + g.z0;
        const double m = (gz > 0 && gz < g.nzg - 1) ? mx : 0.0;
        const double xo = xprev_own;
        double yv;
        if (MODE == M_FIRST2) {
          const double d1 = s0d * xo;
          const double dn = m * fma(a.c1, d1, c2d * fma(-s0d, done, xo));
          yv = m * d1 + dn;
          red_xy = fma(xo, yv, red_xy);
        } else if (CHEBY) {
          const double B = Bv[u];
          const double dprev = a.prev_mode == 1 ? xo - Dv[u]
                             : (a.prev_mode == 2 ? xo : (a.prev_mode == 3 ? xo - s0d * B : 0.0));
          const double dn = m * fma(a.c1, dprev, c2d * (B - done));
          yv = xo + dn;
          red_xy = fma(m * B, yv, red_xy);
        } else {
          yv = m * (HAS_B ? fma(a.ascale, done, a.bscale * Bv[u]) : fma(a.ascale, done, bB));
          red_xy = fma(xo, yv, red_xy);
          red_yy = fma(yv, yv, red_yy);
        }
        if (col && yc) yc[PX * z] = yv;
      }
      xprev_own = v0[u];
    }
  }
  if (a.do_reduce) {
    if (CHEBY) { double v[1] = {red_xy}; block_reduce_finalize<1>(v, red, red_out); }
    else { double v[2] = {red_xy, red_yy}; block_reduce_finalize<2>(v, red, red_out); }
  }
}

static bool sweep2d_applicable(const Grid& g, const OpDev& op, const StencilArgs& a) {
  if (g.dim != 2 || g.nk != 7 || op.ncomp != 1 || !op.uniform_diag) return false;
  if (g.nn[0] < 128 || g.nzl < 8) return false;           // small levels stay on the table kernel (launch bound anyway)
  if (a.ghost_out) return false;
  if (a.cheby == 1 && !a.b) return false;
  return true;
}

template <int MODE>
static int launch_sweep2d_t(pde_ctx* c, const Grid& g, const OpDev& op, const StencilArgs& a) {
  Coef2d C;
  C.c0 = op.h_int[0]; C.cxp = op.h_int[1]; C.cxm = op.h_int[2]; C.czp = op.h_int[5]; C.czm = op.h_int[6];
  C.cdp = op.h_int[9]; C.cdm = op.h_int[10];
  SweepArgs sa;
  sa.x = a.x; sa.b = a.b; sa.y = a.y; sa.xprev = a.xprev; sa.prev_mode = a.prev_mode;
  for (int i = 0; i < 3; ++i) sa.bconst[i] = a.bconst[i];
  sa.bscale = a.bscale; sa.ascale = a.ascale; sa.c1 = a.c1; sa.c2 = a.c2; sa.s0 = a.s0;
  sa.load_int = op.h_load_int;
  for (int i = 0; i < 3; ++i) sa.dinv_int[i] = i < 1 ? op.h_dinv_int[i] : 0.0;
  sa.do_reduce = a.reduce_slot_xy >= 0;
  const int nbx = (g.nn[0] + 255) / 256;
  int zc = 64;
  while (zc > 8 && (long long)nbx * ((g.nzl + zc - 1) / zc) < 4LL * c->sm_count) zc /= 2;
  const int nbz = (g.nzl + zc - 1) / zc;
  if ((long long)nbx * nbz > RED_MAX_BLOCKS) PDE_FAIL("2-D sweep grid exceeds the reduction buffer");
  double* out = sa.do_reduce ? c->scal + a.reduce_slot_xy : nullptr;
  k_sweep2d<MODE><<<(unsigned)(nbx * nbz), 256, 0, c->stream>>>(g, C, sa, zc, nbx, c->red, out);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int launch_elast3d(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a, bool* handled);

// strips of YS = 4 rows for the scalar operators, 2 for the vector ones
template <int NC, int YS>
static int launch_sweep(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a) {
  if (a.cheby == 2) return launch_sweep_t<NC, YS, M_FIRST2>(c, g, bc, op, a);
  if (a.cheby) return launch_sweep_t<NC, YS, M_CHEBY>(c, g, bc, op, a);
  return a.b ? launch_sweep_t<NC, YS, M_RESID>(c, g, bc, op, a) : launch_sweep_t<NC, YS, M_APPLY>(c, g, bc, op, a);
}

int launch_stencil_fast(pde_ctx* c, const Grid& g, const BcDev& bc, const OpDev& op, const StencilArgs& a,
                        bool* handled) {
  *handled = false;
  if (sweep2d_applicable(g, op, a)) {
    *handled = true;
    if (a.cheby == 2) return launch_sweep2d_t<M_FIRST2>(c, g, op, a);
    if (a.cheby) return launch_sweep2d_t<M_CHEBY>(c, g, op, a);
    return a.b ? launch_sweep2d_t<M_RESID>(c, g, op, a) : launch_sweep2d_t<M_APPLY>(c, g, op, a);
  }
  if (!sweep_applicable(g, op.ncomp)) return 0;
  *handled = true;
  if (a.cheby == 1 && !a.b) { *handled = false; return 0; }  // smoother sweeps always carry a rhs field
  if (op.ncomp == 1) return launch_sweep<1, 4>(c, g, bc, op, a);
  if (op.ncomp == 3) {
    // the dedicated elasticity kernel (elast3d.cu) takes the launch when the table has the Kuhn-mesh pattern
    {
      bool h3 = false;
      PDE_OK(launch_elast3d(c, g, bc, op, a, &h3));
      if (h3) return 0;
    }
    // the vector kernel relies on block(+d) == block(-d) for the in-plane pairs and on zero diagonals of the
    // face-/body-diagonal blocks (both structural for P1 elasticity on the Kuhn split); verify, else generic
    double mx = 0;
    for (int q = 0; q < PDE_NOFF * 9; ++q) mx = fmax(mx, fabs(op.h_int[q]));
    bool ok = true;
    const int pairs[3][2] = {{1, 2}, {3, 4}, {7, 8}};
    for (auto& pr : pairs)
      for (int q = 0; q < 9; ++q) ok = ok && fabs(op.h_int[pr[0] * 9 + q] - op.h_int[pr[1] * 9 + q]) <= 1e-12 * mx;
    for (int k = 7; k < PDE_NOFF; ++k)
      for (int i = 0; i < 3; ++i) ok = ok && fabs(op.h_int[k * 9 + i * 3 + i]) <= 1e-12 * mx;
    if (!ok) { *handled = false; return 0; }
    return launch_sweep<3, 2>(c, g, bc, op, a);
  }
  *handled = false;
  return 0;
}
