// kernels.cuh -- launcher declarations shared by capi.cu, eval.cu and solver.cu
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../include/landing_b200.h"
#include "kino_knot.cuh"
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
__host__ __device__ inline long long kino_col(int N, int k, int v) {  // knot-local input v of knot k -> column of x
  if (v < 12) return 12LL * k + v;
  if (v < 24) return 12LL * N + 12LL * k + (v - 12);
  if (v < 48) return 12LL * N + 12LL * (N - 1) + 24LL * k + (v - 24);
  if (v < 60) return 12LL * (k + 1) + (v - 48);
  return 12LL * N + 12LL * (N - 1) + 24LL * (k + 1) + (v - 60);
}
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

// returns number of kernel launches issued
int launch_eval(const EvalArgs& a, cudaStream_t st);
int launch_bounds(const DevicePlan& pl, long long B, CView p, View lbg, View ubg, cudaStream_t st);
int launch_build(const DevicePlan& pl, long long B, const landing_problem& pb, const double* dtv, const double* drops,
                 View p, View x0, cudaStream_t st);

}  // namespace srb
