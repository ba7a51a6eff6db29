// kino_grad.cu -- batched Lagrangian gradient and KKT residuals of the kino-dynamic ("full-body") landing NLP
// (SURVEY 8 f-2): grad_x = lam_f grad f + J' lam_g (CasADi nlp_grad: grad_gamma_x) and, per scenario, the constraint
// violation, the stationarity and the complementarity of a primal-dual point (include/landing_b200.h:
// landing_kino_kkt_batch).  The gradient never forms J: one thread per (scenario, knot, column triple) owns three
// entries of grad_x and runs every Jacobian pass that feeds them (kino_grad.cuh), contracting each dual row with lam_g in
// registers; it writes its three entries once, so there are no atomics, no memset, and every entry is written on every
// call.  The residuals are one thread per scenario over the rows and columns of that scenario.
#include "kernels.cuh"
#include "kino_grad.cuh"

namespace srb {
namespace {

// contraction of an owner: acc[j] += lam_g[row] * dg_row / dz_j.  lam_g is read only for the rows a pass emits as duals.
struct LamCtr {
  CView lam;
  long long b;
  double acc[3];
  __device__ __forceinline__ void operator()(long long row, const kino::DualN<3>& v) {
    const double l = lam.get(row, b);
#pragma unroll
    for (int j = 0; j < 3; j++) acc[j] = fma(l, v.d[j], acc[j]);
  }
  __device__ __forceinline__ void ident(long long row, int j) { acc[j] += lam.get(row, b); }
};

template <int T>
__device__ __forceinline__ void kino_grad_owner(const KinoGradArgs& a, long long b, int k) {
  LamCtr c{a.lam_g, b, {0.0, 0.0, 0.0}};
  const CView x = a.x;
  auto ld = [&](long long col) { return x.get(col, b); };
  if (a.lam_g.p) kino::grad_rows<T>(a.N, k, ld, a.dtv, a.pr, c);
  if (a.lam_f.p) kino::grad_cost<T>(a.N, k, ld, a.lam_f.get(0, b), a.QN, a.ref, c.acc);
#pragma unroll
  for (int j = 0; j < 3; j++) a.grad.at(kino_col(a.N, k, 3 * T + j), b) = c.acc[j];
}
template <int T, int T1>
__device__ __forceinline__ void kino_grad_dispatch(const KinoGradArgs& a, long long b, int k, int t) {
  if constexpr (T < T1) {
    if (t == T) kino_grad_owner<T>(a, b, k);
    else kino_grad_dispatch<T + 1, T1>(a, b, k, t);
  }
}

// Triples T0..T1-1; blockIdx.x = triple + (T1 - T0) * scenario block, blockIdx.y = knot (N knots for the triples of X,
// N - 1 for jpos and U).  One kernel per class of triples (launch_kino_grad), as in k_kino_jac, so that the light passes
// are not held to the register count of the rpy owner (five passes of knot k and the X+ pass of knot k - 1).
template <int T0, int T1, int CTAS>
__global__ void __launch_bounds__(128, CTAS) k_kino_grad(KinoGradArgs a) {
  constexpr int NT = T1 - T0;
  const int t = T0 + (int)(blockIdx.x % NT);
  const long long b = (long long)(blockIdx.x / NT) * 128 + threadIdx.x;
  if (b >= a.B) return;
  kino_grad_dispatch<T0, T1>(a, b, (int)blockIdx.y, t);  // (block-uniform)
}

// One thread per scenario: viol, dual_inf, compl_inf (include/landing_b200.h).  Every input the call was given is read,
// and a NaN in any of them -- or in g or grad_x -- makes every scalar of that scenario NaN (fmax alone would drop it).
__global__ void __launch_bounds__(128) k_kino_kkt(KinoKktArgs a) {
  const long long b = (long long)blockIdx.x * 128 + threadIdx.x;
  if (b >= a.B) return;
  const double INF = HUGE_VAL;
  bool nan = a.lam_f.p && isnan(a.lam_f.get(0, b));
  double viol = 0.0, compl_inf = 0.0, dual = 0.0;
  if (a.g.p || a.lam_g.p || a.lbg.p) {
#pragma unroll 4
    for (long long i = 0; i < a.m; i++) {
      const double gi = a.g.p ? a.g.at(i, b) : 0.0, l = a.lam_g.get(i, b);
      const double lo = a.lbg.p ? a.lbg.get(i, b) : -INF, up = a.lbg.p ? a.ubg.get(i, b) : INF;
      nan = nan || isnan(gi) || isnan(l) || isnan(lo) || isnan(up);
      if (lo > -INF) viol = fmax(viol, lo - gi);
      if (up < INF) viol = fmax(viol, gi - up);
      if (lo < up) {  // inequality rows; a wrong-sign multiplier on an infinite bound gives +inf
        if (l > 0.0) compl_inf = fmax(compl_inf, l * fabs(up - gi));
        else if (l < 0.0) compl_inf = fmax(compl_inf, -l * fabs(gi - lo));
      }
    }
  }
  if (a.grad.p || !a.g.p) {  // (x itself only where no g was computed from it)
#pragma unroll 4
    for (long long j = 0; j < a.nx; j++) {
      const double v = a.grad.p ? a.grad.at(j, b) : 0.0;
      nan = nan || isnan(v) || (!a.g.p && isnan(a.x.get(j, b)));
      dual = fmax(dual, fabs(v));
    }
  }
  const double q = nan ? __longlong_as_double(0x7ff8000000000000LL) : 0.0;
  if (a.viol.p) a.viol.at(0, b) = nan ? q : viol;
  if (a.dual_inf.p) a.dual_inf.at(0, b) = nan ? q : dual;
  if (a.compl_inf.p) a.compl_inf.at(0, b) = nan ? q : compl_inf;
}

}  // namespace

#ifndef KINO_GRAD_CTAS
#define KINO_GRAD_CTAS 6
#endif
#ifndef KINO_GRAD_RPY_CTAS
#define KINO_GRAD_RPY_CTAS 4
#endif
int launch_kino_grad(const KinoGradArgs& a, cudaStream_t st) {
  constexpr int CTAS = KINO_GRAD_CTAS, RPY_CTAS = KINO_GRAD_RPY_CTAS;
  const unsigned gx = (unsigned)((a.B + 127) / 128), nX = a.N, nU = a.N - 1;
  k_kino_grad<0, 1, CTAS><<<dim3(gx * 1, nX, 1), 128, 0, st>>>(a);    // r
  k_kino_grad<1, 2, RPY_CTAS><<<dim3(gx * 1, nX, 1), 128, 0, st>>>(a);    // rpy: dynamics rows and the rows of every leg
  k_kino_grad<2, 4, CTAS><<<dim3(gx * 2, nX, 1), 128, 0, st>>>(a);    // omega, v
  k_kino_grad<4, 8, CTAS><<<dim3(gx * 4, nU, 1), 128, 0, st>>>(a);    // joint angles by leg
  k_kino_grad<8, 12, CTAS><<<dim3(gx * 4, nU, 1), 128, 0, st>>>(a);   // foot positions by leg
  k_kino_grad<12, 16, CTAS><<<dim3(gx * 4, nU, 1), 128, 0, st>>>(a);  // forces by leg
  return 6;
}

int launch_kino_kkt(const KinoKktArgs& a, cudaStream_t st) {
  k_kino_kkt<<<(unsigned)((a.B + 127) / 128), 128, 0, st>>>(a);
  return 1;
}

}  // namespace srb
