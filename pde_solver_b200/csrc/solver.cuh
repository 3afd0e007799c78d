// Solver-layer objects: device fields, operators, multigrid hierarchy, PCG.
#pragma once
#include <functional>
#include <memory>

#include "device.cuh"

struct Field {
  double* raw = nullptr;  // allocation start (ghost plane of component 0)
  double* p = nullptr;    // plane 0 of component 0
  size_t bytes = 0;
  int alloc(pde_ctx* c, const Grid& g, int ncomp);
  void release();
};

struct Operator {
  Grid g{};
  BcDev bc{};
  OpDev dev{};
  OpTable tab;
  int setup_scalar(pde_ctx* c, const Grid& g, const BcDev& bc, double alpha, double beta);
  int setup_elasticity(pde_ctx* c, const Grid& g, const BcDev& bc, double lam, double mu);
  int upload(pde_ctx* c);
  void release();
};

struct MGLevel {
  Operator op;
  Field b, xa, xb, r;
  // slab runs: the level lives on its GLOBAL grid on every rank (no halo exchanges below the first such level);
  // gslab is this rank's window of it (slab z range, global pitch), used when the level above restricts into it
  bool replicated = false;
  Grid gslab{};
  // coarsest level
  int n_dense = 0;
  double* Ainv = nullptr;
  long long* idx = nullptr;   // flat local index of global free dof j (-1: owned by another rank)
  double* bglob = nullptr;    // multi-rank: global coarse right-hand side (all-reduced)
  uint32_t paths = 0;         // PDE_MG_* bits of the fused kernels this level ran (pde_op_vcycle reports them)
};

struct Hierarchy {
  std::vector<std::unique_ptr<MGLevel>> lv;
  int nu = 2;
  double ratio = 8.0;
  int coarse_sweeps = 8;
  // build levels 1.. from a fine operator description; level 0 uses the caller's operator
  int build(pde_ctx* c, const Operator& fine, int kind, double p0, double p1);
  // z = V(b0) ; returns pointer to the buffer holding z (one of level-0 xa/xb)
  // dot_slot >= 0: the last smoother sweep also leaves sum b0.z in that scalar slot if it can (*dot_done)
  int vcycle(pde_ctx* c, const Operator& fine, const double* b0, double** z_out, int dot_slot = -1,
             bool* dot_done = nullptr);
  int levels() const { return (int)lv.size(); }
  void release();
  // single-GPU runs: everything between the level-0 residual and the level-0 post-smoother (restriction, levels
  // 1.., coarsest solve, prolongation into level 0) is a fixed sequence of small kernels with fixed arguments; it is
  // captured into a CUDA graph on the second cycle and replayed afterwards (launch-bound on the coarse levels)
  cudaGraphExec_t gexec = nullptr;
  int gstate = 0;            // 0: no cycle yet, 1: one live cycle done (static set-up complete), 2: graph ready, -1: off
  long long gnodes = 0;      // kernels inside the graph (for the launch count)
};

// First-kind Chebyshev(Jacobi) smoother on [lmax/ratio, lmax]: the recurrence d = c1 d + c2 Dinv r of sweep k
struct Cheby {
  double theta, delta, sigma, rho;
  void init(double lmax, double ratio) {
    const double lmin = lmax / ratio;
    theta = 0.5 * (lmax + lmin);
    delta = 0.5 * (lmax - lmin);
    sigma = theta / delta;
    rho = 1.0 / sigma;
  }
  // coefficients of sweep k (k = 0 restarts the recurrence)
  void coef(int k, double* c1, double* c2) {
    if (k == 0) { rho = 1.0 / sigma; *c1 = 0.0; *c2 = 1.0 / theta; return; }
    const double rn = 1.0 / (2.0 * sigma - rho);
    *c1 = rn * rho;
    *c2 = 2.0 * rn / delta;
    rho = rn;
  }
};

struct PcgWork {
  Field p, q;
  int alloc(pde_ctx* c, const Grid& g, int ncomp);
  void release();
};

// Solves A x = b given x (initial guess incl. Dirichlet values) and r = masked(b - A x).
// bnorm2 = ||b||^2 for the stopping rule ||r|| <= rtol ||b||.  rr0: r.r over all ranks when the caller's
// right-hand-side pass has already formed it (multigrid only; null: computed here).
int pcg_solve(pde_ctx* c, const Operator& A, Hierarchy* mg, PcgWork& w, double* x, double* r, double bnorm2,
              const pde_solver_opts& o, pde_stats* st, const double* rr0 = nullptr);

// The GMG-PCG loop of pcg_solve and wmg_pcg, in the order of oracle/gmg_model.pcg: r -= alpha q is followed by the
// convergence poll, and only an iteration that goes on runs the V-cycle, so a solve of k iterations runs k V-cycles.
// The x update of an iteration rides on its p update (x += alpha p_old, p = z + beta p); the last iteration runs it
// alone.  apply(): q = A p with p.q in S_XY (all-reduced); vcycle(slot, &z): z = V(r) with this rank's r.z in slot.
// rr0 as in pcg_solve.  p, q: work vectors of g.
int mg_pcg(pde_ctx* c, const Grid& g, int ncomp, double* x, double* r, double* p, double* q, double bnorm2,
           const double* rr0, const pde_solver_opts& o, pde_stats* st, const std::function<int()>& apply,
           const std::function<int(int, double**)>& vcycle);

int project_trig_ic(pde_ctx* c, const Grid& g, const BcDev& bc, int dim, const int32_t n_user[3], const double L_user[3],
                    const double* lo_user, double amp, double kw, int use_sin, const pde_solver_opts& o, double* u,
                    double* rhs);
int read_scal(pde_ctx* c, int slot, int count, double* out);
// coarsest multigrid levels with at most this many free dofs are solved with a dense inverse
#define PDE_DENSE_MAX 768
// free dofs of a grid; idx: their flat field indices, dofid: node -> dof number (-1: Dirichlet)
long long count_free_and_index(const Grid& g, const BcDev& bc, int ncomp, std::vector<long long>* idx,
                               std::vector<int>* dofid);
// in-place inverse of a dense SPD matrix (Cholesky); non-zero if it is not positive definite
int dense_inverse_spd(std::vector<double>& A, int n);
int choose_precond(const pde_solver_opts& o, pde_ctx* c, long long ndofs, const Hierarchy& h);
