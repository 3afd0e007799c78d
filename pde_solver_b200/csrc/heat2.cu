// k_heat_post2: the TWO post-smoothing Chebyshev-Jacobi sweeps of the scalar (heat / mass) multigrid levels in ONE pass
// over the data (temporal blocking), for uniform-diagonal operators (every face Dirichlet).
//
//     d0 = m a0 (b - A x0)                         x1 = x0 + d0           (a_k = c2_k / diag, m = 0 on Dirichlet rows)
//     x2 = x1 + m (c1 d0 + a1 (b - A x1))
// On the free rows b - A x0 = d0 / a0, hence b - A x1 = d0 / a0 - A d0 and
//     x2 = x0 + m ((1 + c1 + a1 / a0) d0 - a1 A d0):
// the second sweep is a stencil on d0 alone.  Only ONE field (d0, on the tile grown by one node) goes through the
// shared-memory ring between the two stages; x1 is never formed and b is read once per stage-A node.
//
// Layout (compile time, so that every shared-memory access is base + immediate):
//   tile TX x TY = (CW-2) x 2*YSB nodes (YSB = 4), grown tile CW x (TY+2); a warp covers one row of the grown tile
//   (CW = 64 from 128 nodes in x, else 32), thread = column c of the grown tile x strip s in {0, 1}: stage A owns rows
//   s*YSA + j (YSA = YSB + 1) of the grown tile, stage B rows s*YSB + j of the tile.  Input planes arrive by TMA: x0 as a (TX+4) x (TY+4) box at (x0-2, y0-2), b of the
//   plane stage A retires as a (TX+4) x (TY+2) box at (x0-2, y0-1) in the same pipeline stage (the TMA start coordinate
//   must be 16-byte aligned, hence x0-2).  Stage B runs one plane behind stage A on a three-slot ring of d0 planes and
//   retires x2 one plane later; input planes za-2 .. zb+1 give outputs za .. zb-1 (fields carry PDE_NG = 2 ghost planes).
//   One CTA barrier per plane.
#include <cuda.h>

#include <cmath>

#include "device.cuh"
#include "tma.cuh"

namespace {

// pipeline stages: the post sweeps read the two older stages in stage B (x0 own, b own) and need four; the residual /
// restriction mode only ever reads the current one and runs with three (a fourth CTA per SM fits then)
#ifndef H_RR_STAGES
#define H_RR_STAGES 3
#endif
template <bool RR>
struct HS { static constexpr int N = RR ? H_RR_STAGES : 4; };

template <int CW>
struct HG {
  static constexpr int YSB = 4;
  static constexpr int TX = CW - 2, YSA = YSB + 1, TY = 2 * YSB, RA = TY + 2;
  static constexpr int BX = TX + 4, BYX = TY + 4, BYB = TY + 2;
  static constexpr int XBOX = BX * BYX, BBOX = BX * BYB;              // doubles per TMA box
  static constexpr int XS = (XBOX + 15) / 16 * 16, BS = (BBOX + 15) / 16 * 16;
  static constexpr int STAGE = XS + BS;
  static constexpr int RING = RA * CW;                                // one d0 plane of the grown tile
  static constexpr int NT = 2 * CW;
  static constexpr size_t smem(int nst) { return ((size_t)nst * STAGE + 4 * RING) * sizeof(double) + nst * sizeof(uint64_t); }   // four ring slots
};

struct H2Coef {
  double c0, cxp, cxm, cyp, cym, czp, czm, cxyp, cxym, cxzp, cxzm, cyzp, cyzm, cdp, cdm;   // the 15 offsets, table order
};
struct H2Args {
  double* y;
  double a0, a1, k1;     // k1 = 1 + c1 + a1 / a0
  int do_reduce;
  // RR (residual + restriction): coarse right-hand side (plane 0 of the coarse slab / window) and its grid
  double* yc;
  int cnn0, cnn1, cnzl, cz0, cPX;
  long long cplane;
};
struct H2Geom {
  int nn0, nn1, nzl, z0, nzg, PX;
  long long plane;
  int ntx, nty, nzc, zc;
};

// contributions of one resident plane (values V[r][c]: strip rows r-1, columns c-1) to the outputs one plane below
// (aP: the plane is their dz=+1 neighbour), in the plane (a0) and one plane above (aM: dz=-1, started here)
template <int YS>
__device__ __forceinline__ void h2_contrib(const H2Coef& C, const double (&V)[YS + 2][3], double (&aP)[YS], double (&a0)[YS],
                                           double (&aM)[YS]) {
#pragma unroll
  for (int j = 0; j < YS; ++j) {
    const int r = j + 1;
    double t = fma(C.c0, V[r][1], a0[j]);
    t = fma(C.cxp, V[r][2], t);
    t = fma(C.cxm, V[r][0], t);
    t = fma(C.cyp, V[r + 1][1], t);
    t = fma(C.cym, V[r - 1][1], t);
    t = fma(C.cxyp, V[r + 1][2], t);
    a0[j] = fma(C.cxym, V[r - 1][0], t);
    double p = fma(C.czp, V[r][1], aP[j]);
    p = fma(C.cxzp, V[r][2], p);
    p = fma(C.cyzp, V[r + 1][1], p);
    aP[j] = fma(C.cdp, V[r + 1][2], p);
    double m = C.czm * V[r][1];
    m = fma(C.cxzm, V[r][0], m);
    m = fma(C.cyzm, V[r - 1][1], m);
    aM[j] = fma(C.cdm, V[r - 1][0], m);
  }
}

// RR = false: the two post-smoothing sweeps (above).
// RR = true : residual + restriction in one pass.  Stage A leaves r = m (b - A x) of the grown tile in the ring (a0 = 1) and
//   nothing of it goes to HBM; on every even global plane stage B forms the coarse right-hand side at the even nodes of the
//   tile, r(2X,2Y,2Z) + 1/2 (its 14 Kuhn neighbours), from the three ring planes around it: 17 B per fine dof (x, b in, 1/8
//   out) instead of 24 (residual) + 9 (restriction).  Four ring slots: stage B reads the plane stage A wrote two steps ago.
template <int CW, bool RR>
__global__ void __launch_bounds__(2 * CW, CW == 64 ? ((RR && H_RR_STAGES == 3) ? 4 : 3) : 6)
k_heat_post2(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmb,
             const __grid_constant__ H2Coef C, const __grid_constant__ H2Args a, const __grid_constant__ H2Geom ge,
             ReduceBuf red, double* red_out) {
  using G = HG<CW>;
  constexpr int YSA = G::YSA, YSB = G::YSB;
  constexpr int H_STAGES = HS<RR>::N;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* const stage0 = reinterpret_cast<double*>(smem_raw);
  double* const ring0 = stage0 + H_STAGES * G::STAGE;
  uint64_t* const bars = reinterpret_cast<uint64_t*>(ring0 + 4 * G::RING);

  const int t = threadIdx.x;
  const int item = blockIdx.x;
  const int itx = item % ge.ntx;
  const int ity = (item / ge.ntx) % ge.nty;
  const int izc = item / (ge.ntx * ge.nty);
  const int x0 = itx * G::TX, y0 = ity * G::TY;
  const int za = izc * ge.zc;
  const int zb = min(za + ge.zc, ge.nzl);
  const int nplanes = zb - za + 4;   // x0 planes za-2 .. zb+1
  const uint32_t bar0 = smem_u32(bars);
  const uint32_t stg0 = smem_u32(stage0);
  constexpr uint32_t STAGE_BYTES = G::STAGE * 8;

  // step n: x0 plane za-2+n and (n >= 2) b of the plane stage A retires at that step, za-3+n
  auto issue = [&](int n) {
    const uint32_t bar = bar0 + 8 * (n % H_STAGES);
    const uint32_t dst = stg0 + (n % H_STAGES) * STAGE_BYTES;
    mbar_expect_tx(bar, (uint32_t)((G::XBOX + (n >= 2 ? G::BBOX : 0)) * 8));
    tma_load_4d(dst, &tmx, x0 - 2, y0 - 2, za - 2 + n + PDE_NG, 0, bar);
    if (n >= 2) tma_load_4d(dst + G::XS * 8, &tmb, x0 - 2, y0 - 1, za - 3 + n + PDE_NG, 0, bar);
  };
  if (t == 0) {
#pragma unroll
    for (int s = 0; s < H_STAGES; ++s) mbar_init(bar0 + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (t == 0)
    for (int n = 0; n < 2 && n < nplanes; ++n) issue(n);

  const int c = t % CW;             // column of the grown tile: x = x0 - 1 + c
  const int s = t / CW;             // strip
  const int ix = x0 - 1 + c;
  const int cB = min(max(c, 1), CW - 2);   // stage-B column used for addressing (the two edge columns own no tile node)
  const bool xfree = ix >= 1 && ix <= ge.nn0 - 2;
  unsigned mAb = 0, mBb = 0, okB = 0;      // bit j: stage-A row j free / stage-B row j free / stage-B row j inside the domain
#pragma unroll
  for (int j = 0; j < YSA; ++j) {
    const int iy = y0 - 1 + s * YSA + j;
    if (xfree && iy >= 1 && iy <= ge.nn1 - 2) mAb |= 1u << j;
  }
#pragma unroll
  for (int j = 0; j < YSB; ++j) {
    const int iy = y0 + s * YSB + j;
    const bool in = c >= 1 && c <= G::TX && ix < ge.nn0 && iy < ge.nn1;
    if (in) okB |= 1u << j;
    if (in && xfree && iy >= 1 && iy <= ge.nn1 - 2) mBb |= 1u << j;
  }
  const int offA = (s * YSA) * G::BX + c;                 // x0 box: V[r][cc] = stage[offA + r*BX + cc]
  const int offbA = G::XS + (s * YSA) * G::BX + c + 1;    // b box, stage-A row j: + j*BX
  const int offbB = G::XS + (s * YSB + 1) * G::BX + cB + 1;   // b box, stage-B row j: + j*BX
  const int offxB = (s * YSB + 2) * G::BX + cB + 1;       // x0 box, stage-B row j (own node): + j*BX
  const int ringA = (s * YSA) * CW + c;                   // d0 plane, stage-A row j: + j*CW
  const int ringB = (s * YSB) * CW + cB - 1;              // d0 plane: VB[r][cc] = ring[ringB + r*CW + cc]
  double* yrun = a.y + ((long long)ge.PX * (y0 + s * YSB) + ix) + ge.plane * za;   // output column at plane za

  double aA[YSA], aB[YSA], aC[YSA];        // stage-A accumulators (three planes in flight)
  double bA_[YSB], bB_[YSB], bC_[YSB];     // stage-B accumulators
#pragma unroll
  for (int j = 0; j < YSA; ++j) aA[j] = aB[j] = aC[j] = 0.0;
#pragma unroll
  for (int j = 0; j < YSB; ++j) bA_[j] = bB_[j] = bC_[j] = 0.0;
  double red_by = 0.0;

  auto body = [&](int i, double (&aP)[YSA], double (&a0)[YSA], double (&aM)[YSA], double (&bP)[YSB], double (&b0)[YSB],
                  double (&bM)[YSB]) {
    const int stage = i % H_STAGES;
    const int q = za - 2 + i;          // resident x0 plane
    const int pA = q - 1;              // plane stage A retires (d0)
    const int pB = q - 2;              // plane stage B retires (x2)
    const bool finA = i >= 2, finB = i >= 4;
    // what stage B needs of older pipeline stages is read before the barrier, so that stage i-2 can be refilled after it
    double xB0[YSB], bvB[YSB];
    if (!RR && finB) {
      const double* const sx2 = stage0 + ((i - 2) % H_STAGES) * G::STAGE + offxB;
      const double* const sb1 = stage0 + ((i - 1) % H_STAGES) * G::STAGE + offbB;
#pragma unroll
      for (int j = 0; j < YSB; ++j) { xB0[j] = sx2[j * G::BX]; bvB[j] = sb1[j * G::BX]; }
    }
    mbar_wait(bar0 + 8 * stage, (uint32_t)((i / H_STAGES) & 1));
    const double* const sx = stage0 + stage * G::STAGE;
    {  // ---- stage A: plane q of x0 ----
      double V[YSA + 2][3];
      const double* const sp = sx + offA;
#pragma unroll
      for (int r = 0; r < YSA + 2; ++r)
#pragma unroll
        for (int cc = 0; cc < 3; ++cc)
          V[r][cc] = ((r == 0 && cc == 2) || (r == YSA + 1 && cc == 0)) ? 0.0 : sp[r * G::BX + cc];
      h2_contrib<YSA>(C, V, aP, a0, aM);
    }
    if (finA) {
      const int gz = pA + ge.z0;
      const bool zfree = gz >= 1 && gz <= ge.nzg - 2;
      const unsigned mA = zfree ? mAb : 0u;
      double* const ds = ring0 + ((pA + 4) & 3) * G::RING + ringA;
      const double* const sb = sx + offbA;
#pragma unroll
      for (int j = 0; j < YSA; ++j) ds[j * CW] = ((mA >> j) & 1u) ? a.a0 * (sb[j * G::BX] - aP[j]) : 0.0;
    }
    __syncthreads();   // plane pA of d0 is visible; stage i-2 (and the reads of stage B above) are done
    if (t == 0 && i + 2 < nplanes) issue(i + 2);
    if (!RR && finA) {  // ---- stage B: plane pA of d0 ----
      double V[YSB + 2][3];
      const double* const rp = ring0 + ((pA + 4) & 3) * G::RING + ringB;
#pragma unroll
      for (int r = 0; r < YSB + 2; ++r)
#pragma unroll
        for (int cc = 0; cc < 3; ++cc)
          V[r][cc] = ((r == 0 && cc == 2) || (r == YSB + 1 && cc == 0)) ? 0.0 : rp[r * CW + cc];
      h2_contrib<YSB>(C, V, bP, b0, bM);
    }
    if (RR && finB) {
      // ---- restriction: coarse plane Z = (pB + z0) / 2 from the residual planes pB-1, pB, pB+1 (= pA) of the ring ----
      const int gz = pB + ge.z0;
      const int Z = (gz >> 1) - a.cz0;
      constexpr int NCX = G::TX / 2, NCY = G::TY / 2;
      if (!(gz & 1) && Z >= 0 && Z < a.cnzl && t < NCX * NCY) {
        const int cx = t % NCX, cy = t / NCX;
        const int X = (x0 >> 1) + cx, Y = (y0 >> 1) + cy;
        if (X < a.cnn0 && Y < a.cnn1) {
          const int o = (1 + 2 * cy) * CW + 1 + 2 * cx;      // the fine node in the grown tile
          const double* const r0 = ring0 + ((pB + 4) & 3) * G::RING + o;
          const double* const rm = ring0 + ((pB + 3) & 3) * G::RING + o;
          const double* const rp = ring0 + ((pB + 5) & 3) * G::RING + o;
          const double nb = ((r0[1] + r0[-1]) + (r0[CW] + r0[-CW])) + ((r0[CW + 1] + r0[-CW - 1]) + (rp[0] + rm[0])) +
                            ((rp[1] + rm[-1]) + (rp[CW] + rm[-CW])) + (rp[CW + 1] + rm[-CW - 1]);
          const int cgz = gz >> 1;
          const bool cfree = X >= 1 && X <= a.cnn0 - 2 && Y >= 1 && Y <= a.cnn1 - 2 && cgz >= 1 && cgz <= (ge.nzg >> 1) - 1;
          a.yc[(long long)a.cPX * Y + a.cplane * Z + X] = cfree ? fma(0.5, nb, r0[0]) : 0.0;
        }
      }
    }
    if (!RR && finB) {
      const int gz = pB + ge.z0;
      const bool zfree = gz >= 1 && gz <= ge.nzg - 2;
      const unsigned mB = zfree ? mBb : 0u;
      const double* const dso = ring0 + ((pB + 4) & 3) * G::RING + ringB + CW + 1;   // own node of stage-B row j: + j*CW
#pragma unroll
      for (int j = 0; j < YSB; ++j) {
        const bool m = (mB >> j) & 1u;
        const double x2 = m ? fma(a.k1, dso[j * CW], fma(-a.a1, bP[j], xB0[j])) : xB0[j];
        if ((okB >> j) & 1u) yrun[j * (long long)ge.PX] = x2;
        red_by = fma(m ? bvB[j] : 0.0, x2, red_by);
      }
      yrun += ge.plane;
    }
  };

  // stage-A roles rotate from step 0, stage-B roles from step 2 (its first plane)
  for (int i = 0; i < nplanes; i += 3) {
    body(i, aA, aB, aC, bB_, bC_, bA_);
    if (i + 1 < nplanes) body(i + 1, aB, aC, aA, bC_, bA_, bB_);
    if (i + 2 < nplanes) body(i + 2, aC, aA, aB, bA_, bB_, bC_);
  }
  if (a.do_reduce) {
    double v[1] = {red_by};
    block_reduce_finalize<1>(v, red, red_out);
  }
}

template <int CW, bool RR>
int launch_t(pde_ctx* c, const Grid& g, const OpDev& op, const double* x0, const double* b, const H2Args& ha_in) {
  using G = HG<CW>;
  H2Geom ge;
  ge.nn0 = g.nn[0]; ge.nn1 = g.nn[1]; ge.nzl = g.nzl; ge.z0 = g.z0; ge.nzg = g.nzg; ge.PX = g.PX; ge.plane = g.plane;
  ge.ntx = (g.nn[0] + G::TX - 1) / G::TX;
  ge.nty = (g.nn[1] + G::TY - 1) / G::TY;
  int zc = 64;
  while (zc > 8 && (long long)ge.ntx * ge.nty * ((g.nzl + zc - 1) / zc) < 6LL * c->sm_count) zc /= 2;
  // grids thin in x have many tiles per plane (33 x 4097 x 4097 nodes: 1026): longer z chunks keep the grid within the
  // reduction buffer
  while (zc < g.nzl && (long long)ge.ntx * ge.nty * ((g.nzl + zc - 1) / zc) > RED_MAX_BLOCKS) zc *= 2;
  ge.nzc = (g.nzl + zc - 1) / zc;
  ge.zc = (g.nzl + ge.nzc - 1) / ge.nzc;
  ge.nzc = (g.nzl + ge.zc - 1) / ge.zc;
  const long long items = (long long)ge.ntx * ge.nty * ge.nzc;
  if (items > RED_MAX_BLOCKS) return 2;   // the tiles of one plane alone exceed it: the caller falls back
  auto kern = k_heat_post2<CW, RR>;
  static bool attr_set = false;
  if (!attr_set) {
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::smem(HS<RR>::N)));
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    attr_set = true;
  }
  CUtensorMap tmx, tmb;
  PDE_OK(field_tensor_map(x0, g, 1, G::BX, G::BYX, &tmx));
  PDE_OK(field_tensor_map(b, g, 1, G::BX, G::BYB, &tmb));
  H2Coef C;
  const double* h = op.h_int;
  C.c0 = h[0]; C.cxp = h[1]; C.cxm = h[2]; C.cyp = h[3]; C.cym = h[4]; C.czp = h[5]; C.czm = h[6]; C.cxyp = h[7];
  C.cxym = h[8]; C.cxzp = h[9]; C.cxzm = h[10]; C.cyzp = h[11]; C.cyzm = h[12]; C.cdp = h[13]; C.cdm = h[14];
  kern<<<(unsigned)items, G::NT, G::smem(HS<RR>::N), c->stream>>>(tmx, tmb, C, ha_in, ge, c->red, ha_in.do_reduce ? c->scal + ha_in.do_reduce - 1 : nullptr);
  c->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

template <bool RR>
int dispatch(pde_ctx* c, const Grid& g, const OpDev& op, const double* x0, const double* b, const H2Args& ha) {
  if (g.nn[0] >= 128) return launch_t<64, RR>(c, g, op, x0, b, ha);
  return launch_t<32, RR>(c, g, op, x0, b, ha);
}

}  // namespace

// does k_heat_post2 (both post-smoothing sweeps, or residual + restriction) take this level?
bool heat2_applicable(const Grid& g, const OpDev& op) {
  if (g.dim != 3 || g.nk != PDE_NOFF || op.ncomp != 1 || !op.uniform_diag) return false;
  return g.nn[0] >= 32 && g.nn[1] >= 8 && g.nzl >= 8;
}

// Two restart Chebyshev sweeps in one pass; *handled = false if the kernel does not apply (the caller falls back).
int launch_heat_post2(pde_ctx* c, const Grid& g, const OpDev& op, const double* x0, const double* b, double* y, double c2_0,
                      double c1_1, double c2_1, int dot_slot, bool* handled) {
  *handled = false;
  if (!heat2_applicable(g, op) || !(c2_0 * op.h_dinv_int[0] > 0.0)) return 0;
  H2Args ha{};
  ha.y = y;
  ha.a0 = c2_0 * op.h_dinv_int[0];
  ha.a1 = c2_1 * op.h_dinv_int[0];
  ha.k1 = 1.0 + c1_1 + ha.a1 / ha.a0;
  ha.do_reduce = dot_slot >= 0 ? dot_slot + 1 : 0;   // slot + 1 (0: none)
  const int rc = dispatch<false>(c, g, op, x0, b, ha);
  if (rc == 0) *handled = true;
  return rc == 2 ? 0 : rc;
}

// Residual of level gf and its restriction into the coarse grid gc (a slab, or this rank's window of a replicated
// level) in one pass: bcoarse = R (b - A x), the fine residual is never stored.  Needs two valid halo planes of x and
// one of b on slab runs (the lean halo scheme provides them).
int launch_heat_resid_restrict(pde_ctx* c, const Grid& gf, const Grid& gc, const OpDev& op, const double* x, const double* b,
                               double* bcoarse, bool* handled) {
  *handled = false;
  if (!heat2_applicable(gf, op)) return 0;
  // nested grids, slab windows that nest too (rank r owns coarse planes z0/2 ...)
  if (gf.nc[0] != 2 * gc.nc[0] || gf.nc[1] != 2 * gc.nc[1] || gf.nc[2] != 2 * gc.nc[2] || gf.z0 != 2 * gc.z0) return 0;
  H2Args ha{};
  ha.a0 = 1.0;
  ha.yc = bcoarse;
  ha.cnn0 = gc.nn[0]; ha.cnn1 = gc.nn[1]; ha.cnzl = gc.nzl; ha.cz0 = gc.z0; ha.cPX = gc.PX; ha.cplane = gc.plane;
  const int rc = dispatch<true>(c, gf, op, x, b, ha);
  if (rc == 0) *handled = true;
  return rc == 2 ? 0 : rc;
}
