// tests/hostcheck/kino_step_host.cpp -- TEST HARNESS (CPU): compiles the interior-point Newton step of the kino-dynamic
// NLP (landing_controller_b200/csrc/kino_step.cuh: the plan, the Riccati sweeps, the recovery and the inertia schedule)
// for the host, as a team of one thread, so that it can be checked against a dense solve of the full system without a
// GPU.  Not part of the product library and never used as a fallback.
#include <vector>

#include "../../landing_controller_b200/csrc/kino_step.cuh"

using namespace srb::kino;

struct HostIn {
  const double *J, *H, *G;
  double jac(long long i) const { return J[i]; }
  double hess(long long i) const { return H[i]; }
  double gf(long long i) const { return G[i]; }
};
// instrumented source: how often the assembly reads each entry
struct CountIn {
  const double *J, *H, *G;
  int *jc, *hc, *gc;
  double jac(long long i) const { jc[i]++; return J[i]; }
  double hess(long long i) const { hc[i]++; return H[i]; }
  double gf(long long i) const { gc[i]++; return G[i]; }
};

static StepTables view(const KinoStepPlan& p) {
  return StepTables{p.N, p.nx, p.m, p.mstage.data(), p.mtgt.data(), p.mbeg.data(), p.mterm.data(), p.qstage.data(),
                    p.qtgt.data(), p.qbeg.data(), p.qterm.data(), p.dstage.data(), p.dterm.data(), p.rptr.data(),
                    p.rent.data()};
}
static KinoStepPlan plan(int N, const long long* jsp, const long long* hsp) {
  const long long nx = jsp[1];
  return make_kino_step_plan(N, jsp + 2, jsp + 2 + nx + 1, hsp + 2, hsp + 2 + nx + 1);
}

// One scenario.  vec: g, s, y, zL, zU, lbg, ubg [m]; out5: dx [nx], ds, dy, dzL, dzU [m]; res: delta_w, n_factor,
// status, alpha_pr, alpha_du.  Returns -1 if the plan is refused.
extern "C" int kino_step_host(int N, const long long* jsp, const long long* hsp, const double* jac, const double* hess,
                              const double* grad_f, const double* const* vec, double mu, double dw_last, double tau,
                              double* const* out5, double* res) {
  const KinoStepPlan pl = plan(N, jsp, hsp);
  if (!pl.err.empty()) return -1;
  const StepTables tb = view(pl);
  const HostIn in{jac, hess, grad_f};
  const StepPoint it{{vec[0], 1}, {vec[1], 1}, {vec[2], 1}, {vec[3], 1}, {vec[4], 1}, {vec[5], 1}, {vec[6], 1}, mu};
  const StepOut o{{out5[0], 1}, {out5[1], 1}, {out5[2], 1}, {out5[3], 1}, {out5[4], 1}};
  std::vector<double> smem(STEP_SMEM), scr((size_t)N * STEP_STAGE);
  StepShared sh(smem.data());
  const Team tm{0, 1};
  if (!step_interior(it, tb.m, tm)) {
    res[2] = 5;  // LANDING_ST_NOT_INTERIOR
    return 0;
  }
  double dw = dw_first(dw_last);
  int nf = 0, status = 0;
  for (int tries = 0;;) {
    nf++;
    if (step_factor(tb, in, it, dw, sh, scr.data(), tm)) break;
    dw = dw_next(dw, dw_last, tries);
    tries++;
    if (dw > 1e40) { status = 4; break; }
  }
  res[0] = dw; res[1] = nf; res[2] = status;
  if (status == 0) step_solve(tb, in, it, scr.data(), sh, o, tau, &res[3], &res[4], tm);
  return 0;
}

// Coverage of one factorisation with dw: jcnt [nnzJ], hcnt [nnzH], gcnt [nx] count the reads of each entry by the
// stage assembly (zeroed by the caller); jrole [nnzJ] is the plan's role of each Jacobian entry (0 boundary identity,
// 1 identity on X_{k+1}, 2 dynamics, 3 inequality row).  Returns -1 if the plan is refused.
extern "C" int kino_step_cover(int N, const long long* jsp, const long long* hsp, const double* jac, const double* hess,
                               const double* grad_f, const double* const* vec, double mu, int* jcnt, int* hcnt, int* gcnt,
                               int* jrole) {
  const KinoStepPlan pl = plan(N, jsp, hsp);
  if (!pl.err.empty()) return -1;
  for (size_t e = 0; e < pl.jrole.size(); e++) jrole[e] = pl.jrole[e];
  const StepTables tb = view(pl);
  const CountIn in{jac, hess, grad_f, jcnt, hcnt, gcnt};
  const StepPoint it{{vec[0], 1}, {vec[1], 1}, {vec[2], 1}, {vec[3], 1}, {vec[4], 1}, {vec[5], 1}, {vec[6], 1}, mu};
  std::vector<double> smem(STEP_SMEM);
  StepShared sh(smem.data());
  for (int k = N - 1; k >= 0; k--) assemble_stage(tb, k, in, it, 0.0, sh, Team{0, 1});
  return 0;
}

// The plan's verdict on a pattern (for refused patterns): 0 accepted, -1 refused.
extern "C" int kino_step_plan_ok(int N, const long long* jsp, const long long* hsp) { return plan(N, jsp, hsp).err.empty() ? 0 : -1; }
