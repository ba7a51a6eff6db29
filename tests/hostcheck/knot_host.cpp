// tests/hostcheck/knot_host.cpp -- TEST HARNESS (CPU): compiles the product's knot template
// (landing_controller_b200/csrc/srb_knot.cuh, plan.cuh) for the host so that the kernel math and
// the CCS scatter maps can be checked against the oracle without a GPU.  Not part of the product
// library and never used as a fallback.
#include <cstring>
#include "../../landing_controller_b200/csrc/plan.cuh"

using namespace srb;

struct HostSink {
  double *gv, *jac, *hes;
  const int *jm, *hm;
  void g(int row, double v) { if (gv) gv[row] = v; }
  void j(int e, int, int, double v) { if (jac) jac[jm[e]] = v; }
  void h(int e, int, int, double v) { if (hes) hes[hm[e]] = v; }
};
struct HostLam {
  const double* l;
  double operator()(int row) const { return l ? l[row] : 0.0; }
};

// cs == nullptr: formulation 0; else the SCHED instantiation (formulation 1) with cs[4 k + leg] of knot k
static int eval_all(int N, const double* x, const double* p, double lam_f, const double* lam_g, const int* cs,
                    double* g, double* jac, double* hes) {
  auto pl = get_plan(N);
  const ParamOff& o = pl->off;
  if (g) {
    for (int i = 0; i < 12; i++) g[i] = x[i];
    for (int i = 0; i < 6; i++) {
      g[12 + i] = g[18 + i] = x[12 * (N - 1) + i];
      g[24 + i] = g[30 + i] = x[12 * (N - 1) + 6 + i];
    }
  }
  if (jac) for (int i = 0; i < 36; i++) jac[pl->jbnd[i]] = 1.0;
  if (hes) for (int i = 0; i < 12; i++) hes[pl->hterm[i]] = 2.0 * p[o.QN + i] * lam_f;
  for (int k = 0; k < N - 1; k++) {
    Knot kn;
    const bool last = k == N - 2;
    for (int i = 0; i < 12; i++) {
      kn.X[i] = x[12 * k + i];
      kn.Xn[i] = x[12 * (k + 1) + i];
      kn.c[i] = x[12 * N + 24 * k + i];
      kn.f[i] = x[12 * N + 24 * k + 12 + i];
      kn.cn[i] = last ? 0.0 : x[12 * N + 24 * (k + 1) + i];
    }
    kn.h = p[o.dt + k]; kn.mu = p[o.mu]; kn.mass = p[o.mass];
    for (int i = 0; i < 3; i++) { kn.Ib[i] = p[o.Ib + i]; kn.Ibinv[i] = p[o.Ibinv + i]; }
    for (int l = 0; l < 4; l++) kn.csv[l] = cs ? (double)cs[4 * k + l] : 0.0;
    HostSink s{g ? g + 36 + 104 * k : nullptr, jac, hes, pl->jmap.data() + k * NJ_INT, pl->hmap.data() + k * NH_INT};
    HostLam lam{lam_g ? lam_g + 36 + 104 * k : nullptr};
    if (cs) {
      if (last) knot_eval<true, true, true, true, HostSink, HostLam, true>(kn, s, lam);
      else knot_eval<false, true, true, true, HostSink, HostLam, true>(kn, s, lam);
    } else {
      if (last) knot_eval<true, true, true, true>(kn, s, lam);
      else knot_eval<false, true, true, true>(kn, s, lam);
    }
  }
  return 0;
}
extern "C" int hostcheck_eval(int N, const double* x, const double* p, double lam_f, const double* lam_g,
                              double* g, double* jac, double* hes) {
  return eval_all(N, x, p, lam_f, lam_g, nullptr, g, jac, hes);
}
// the fixed-contact-schedule instantiation; the boundary rows 0..35 are filled as in hostcheck_eval
extern "C" int hostcheck_eval_sched(int N, const double* x, const double* p, double lam_f, const double* lam_g,
                                    const int* cs, double* g, double* jac, double* hes) {
  return eval_all(N, x, p, lam_f, lam_g, cs, g, jac, hes);
}
extern "C" const long long* hostcheck_sparsity(int N, int which) {
  auto pl = get_plan(N);
  return which == 0 ? pl->spJ.data() : pl->spH.data();
}
