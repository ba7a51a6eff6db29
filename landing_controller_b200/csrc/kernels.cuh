// kernels.cuh -- launcher declarations shared by capi.cu, eval.cu and solver.cu
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../include/landing_b200.h"
#include "kino_knot.cuh"
#include "kino_step.cuh"
#include "plan.cuh"

namespace srb {

// strided view of a [n x B] family of per-scenario vectors: element i of scenario b at p[i*si + b*sb]
struct View {
  double* p;
  long long si, sb;
  __host__ __device__ __forceinline__ double& at(long long i, long long b) const { return p[i * si + b * sb]; }
};
struct CView {
  const double* p;
  long long si, sb;
  __host__ __device__ __forceinline__ double get(long long i, long long b) const {
    return p ? p[i * si + b * sb] : 0.0;  // NULL input == all zeros (landingCtrller_IPOPT.c:69)
  }
};

inline View make_view(double* p, long long n, long long B, int layout) {
  return layout == LANDING_SOA ? View{p, B, 1} : View{p, 1, n};
}
inline CView make_cview(const double* p, long long n, long long B, int layout) {
  return layout == LANDING_SOA ? CView{p, B, 1} : CView{p, 1, n};
}

struct DevicePlan {  // device copies of the scatter maps
  int N, nx, np, m, nnzJ, nnzH;
  ParamOff off;
  const int *jmap, *hmap, *jbnd, *hterm;
};

struct EvalArgs {
  DevicePlan pl;
  long long B;
  CView x, p, lam_f, lam_g;
  View f, g, grad_f, jac, hess, grad_x, grad_p;
  int* status;
  int k0 = 0;  // first knot slice handled by blockIdx.y == 0
};

// dst[c][r] = src[r][c] for a row-major rows x cols matrix of doubles (32 x 32 shared-memory tiles); returns 1
int launch_transpose(const double* src, double* dst, long long rows, long long cols, cudaStream_t st);

struct TvlqrArgs {
  int N;
  long long nx;
  const double* x_star;  // [B][nx] solved trajectories (AoS)
  double *P_out, *K_out; // [B][n_steps][24*24], [B][n_steps][12*24] (either may be null)
  landing_tvlqr par;
};
int launch_tvlqr(const TvlqrArgs& a, long long B, cudaStream_t st);

// kino-dynamic NLP (kino.cu): host plan (sizes, CCS pattern, scatter tables) and the batched evaluation
__host__ __device__ inline long long kino_col(int N, int k, int v) { return kino::knot_col(N, k, v); }
struct KinoPlan {
  int N = 0;
  long long nx = 0, m = 0, nnz = 0;
  std::vector<long long> sparsity;  // CasADi CCS {nrow, ncol, colind[ncol+1], row[nnz]}
  std::vector<int> gpos;            // [knot][local input 72][local row 141] -> CCS position or -1
  std::vector<int> bpos;            // the 48 boundary rows' (identity) entries
};
KinoPlan make_kino_plan(int N);
struct KinoArgs {
  int N;
  long long B;
  CView x;
  View g, jac;
  kino::Params pr;
  const double* dtv;  // knot spacings (device)
  const int *gpos, *bpos;
};
int launch_kino(const KinoArgs& a, bool want_g, bool want_jac, cudaStream_t st);
struct KinoSetupArgs {
  int N;
  long long B;
  landing_kino_setup ks;
  CView drops, x_srb;  // [12 x B]; [36N-24 x B] or null
  View lbg, ubg, x0;   // any may be null
  CView x;             // cost: [n_x x B]
  View f, grad_f;
};
int launch_kino_setup(const KinoSetupArgs& a, cudaStream_t st);
int launch_kino_cost(const KinoSetupArgs& a, cudaStream_t st);
// Lagrangian Hessian of the kino-dynamic NLP (kino_hess.cu): upper-triangle CCS pattern and the writer of every entry
struct KinoHessPlan {
  int N = 0;
  long long nx = 0, nnz = 0;
  std::vector<long long> sparsity;  // CasADi CCS {nx, nx, colind[nx+1], row[nnz]}, upper triangle
  std::vector<int> hpos;            // [knot][pass][3 x 3] -> CCS position or -1
  std::vector<unsigned> rows;       // [knot class][pass][5 words]: rows with a second-order part in the pass's block
  std::vector<int> cpos;            // [12] terminal-cost diagonal of X_{N-1}
  std::string err;                  // non-empty: the pair table misses a non-zero block, or an entry has two writers
};
KinoHessPlan make_kino_hess_plan(int N);
struct KinoHessArgs {
  int N;
  long long B;
  CView x, lam_f, lam_g;
  View hess;
  kino::Params pr;
  double QN[12];      // 0 without lam_f
  const double* dtv;  // knot spacings (device)
  const int *hpos, *cpos;
  const unsigned* rows;
};
int launch_kino_hess(const KinoHessArgs& a, cudaStream_t st);
// Lagrangian gradient and KKT residuals of the kino-dynamic NLP (kino_grad.cu)
struct KinoGradArgs {
  int N;
  long long B;
  CView x, lam_f, lam_g;  // lam_f / lam_g NULL: no cost / no row terms
  View grad;
  kino::Params pr;
  double QN[12], ref[12];  // terminal cost (with lam_f)
  const double* dtv;       // knot spacings (device)
};
int launch_kino_grad(const KinoGradArgs& a, cudaStream_t st);
struct KinoKktArgs {
  long long B, m, nx;
  CView x, lam_f, lam_g, lbg, ubg;  // any may be NULL but x
  View g, grad;                     // g(x) when viol / compl_inf are wanted, grad_x when dual_inf is; else NULL
  View viol, dual_inf, compl_inf;   // [1 x B], any may be NULL
};
int launch_kino_kkt(const KinoKktArgs& a, cudaStream_t st);
// interior-point Newton step of the kino-dynamic NLP (kino_step.cu): the plan's tables (one flat int array, offsets of
// the twelve StepTables arrays) and the launch
struct KinoStepHost {
  int N = 0;
  long long nx = 0, m = 0, off[12] = {};
  std::vector<int> flat;
};
std::string make_kino_step_tables(int N, const long long* jac_sparsity, const long long* hess_sparsity, KinoStepHost* out);
kino::StepTables kino_step_view(const KinoStepHost& h, const int* dev);
struct KinoStepArgs {
  long long B;
  kino::StepTables tb;
  CView g, jac, hess, grad_f, s, y, zL, zU, lbg, ubg, mu, dw_last;
  View dx, ds, dy, dzL, dzU, delta_w, alpha_pr, alpha_du;  // alpha_*: p NULL when not wanted
  int *n_factor, *status;  // [B]
  double tau;
  double* scratch;  // [grid][slot]
  long long slot;
  int* counter;     // scenario counter (zeroed before the launch)
};
int kino_step_smem_bytes();
long long kino_step_slot(int N);
int kino_step_resident(cudaError_t* err);
int launch_kino_step(const KinoStepArgs& a, int grid, cudaStream_t st);

// returns number of kernel launches issued
int launch_eval(const EvalArgs& a, cudaStream_t st);
int launch_bounds(const DevicePlan& pl, long long B, CView p, View lbg, View ubg, cudaStream_t st);
int launch_build(const DevicePlan& pl, long long B, const landing_problem& pb, const double* dtv, const double* drops,
                 View p, View x0, cudaStream_t st);

}  // namespace srb
