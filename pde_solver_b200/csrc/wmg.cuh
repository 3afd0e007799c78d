// Galerkin geometric multigrid for the per-node (weighted) operators of weighted.cu.
#pragma once
#include "solver.cuh"

// Flat offsets of the stored half of the Kuhn stencil: plane 0 is the centre, plane j >= 1 holds a(i, i + off[j]) for
// the positive member of the j-th +/- offset pair; the partner a(i, i - off[j]) is read at the neighbour.
struct WStencil {
  int nh;             // stored planes: 8 (3-D), 4 (2-D), 2 (1-D)
  long long off[8];
  int dx[8], dy[8], dz[8];
  int kidx[27];       // (dx+1) + 3(dy+1) + 9(dz+1) -> index into g.kdx/kdy/kdz, -1 outside the stencil
};

struct WLevel {
  Grid g{};
  WStencil ws{};
  Field h;            // nh planes of symmetric half coefficients, Dirichlet rows and columns zero
  Field b, xa, xb, r;
  double lmax = 0.0;  // Gershgorin bound of D^-1 A
  int n_dense = 0;    // coarsest level: dense inverse over the free nodes
  double* Ainv = nullptr;
  long long* idx = nullptr;
};

struct WHierarchy {
  std::vector<std::unique_ptr<WLevel>> lv;
  BcDev bc{};
  int nu = 2;
  double ratio = 8.0;
  int coarse_sweeps = 8;
  // Level 0 from the full stencil coefA (g.nk planes); coarser levels are P^T A P while every axis halves evenly.
  // One level only: the grid does not coarsen and the caller runs Jacobi-PCG instead.
  int build(pde_ctx* c, const Grid& g0, const BcDev& bc0, const double* coefA);
  int levels() const { return (int)lv.size(); }
  void release();
  ~WHierarchy() { release(); }
};

// GMG-PCG on A x = b given x (with Dirichlet values) and r = masked(b - A x); p, q: work vectors of level 0's grid
int wmg_pcg(pde_ctx* c, WHierarchy& h, double* x, double* r, double* p, double* q, double bnorm2,
            const pde_solver_opts& o, pde_stats* st);
// z = V(b0) (z_out: the level-0 buffer holding it); the last level-0 post-sweep leaves sum b0.z in dot_slot
int wvcycle(pde_ctx* c, WHierarchy& H, const double* b0, double** z_out, int dot_slot);
// level `level` expanded to all g.nk offsets (g.kdx order), [nk][nverts] in natural vertex order
int wmg_level_coefs(pde_ctx* c, const WHierarchy& h, int level, double* out);
