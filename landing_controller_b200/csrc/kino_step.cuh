// kino_step.cuh -- the primal-dual Newton step of one interior-point iteration of the kino-dynamic NLP, host and device
// (include/landing_b200.h: landing_kino_step_batch).  IPOPT's form, as oracle/ip_ref.c: slacks s on the inequality rows,
// bound multipliers zL / zU on their finite bounds, y with CasADi's sign (L = f + y'(g - s)), W the Lagrangian Hessian
// with lam_f = 1 and lam_g = y.  Slacks and bound multipliers are eliminated (sigma = zL / (s - lbg) + zU / (ubg - s) on
// each inequality row), which leaves the equality-constrained QP in dx
//   min 1/2 dx' (W + J_I' Sigma J_I + dw I) dx + (grad f + J_I' yhat)' dx   s.t.   J_E dx = -(g_E - lbg_E),
// solved by a Riccati recursion over the stages of the knots:
//   stage k (k = 0..N-2): 60 variables, the state xi_k = (X_k, c_k) (stage columns 0..23) and the control
//     u_k = (jpos_k, f_k, c_{k+1}) (24..59; the last stage has no c_{N-1}: its columns 48..59 are a decoupled identity);
//   stage N-1 (terminal): X_{N-1} in columns 0..11.
// The rows of knot k other than its 12 dynamics rows reach only the variables of stage k, the terminal rows 24..47 only
// X_{N-1}; the dynamics rows give X_{k+1} = G_k (X_k, c_k, f_k) + r_k (coefficient 1 on X_{k+1}); the boundary rows 0..23
// fix xi_0.  X_0 and c_0 are both fixed, so the null space of J_E is parametrised by the controls alone and "every control
// block has a Cholesky pivot > 1e-14" is exactly "the reduced Hessian is positive definite": the inertia test.
//
// Everything here is written for a team of threads (one CTA per scenario on the device, one thread on the host): loops
// stride over the team and team_sync() separates the phases, so the host build (tests/hostcheck/kino_step_host.cpp) runs
// the same code.  Every sum has a fixed order, so the result does not depend on the team size's scheduling.
#pragma once
#include <cmath>

#include <algorithm>
#include <string>
#include <vector>

#include "kino_knot.cuh"

namespace srb {
namespace kino {

constexpr int SW = 60, SXI = 24, SU = 36;  // stage width, state, control

struct Team {
  int tid, nt;
};
KHD void team_sync() {
#ifdef __CUDA_ARCH__
  __syncthreads();
#endif
}

// structural row kinds: the boundary rows 0..23 and the 12 dynamics rows of each knot are the equality rows
KHD bool step_is_eq(long long row) { return row < 24 || (row >= 48 && (row - 48) % ROWS_INT < 12); }
// dynamics row rho (v, omega, r, rpy) -> state index (r, rpy, omega, v)
KHD int dynrow_state(int rho) { return rho < 3 ? 9 + rho : rho < 6 ? 3 + rho : rho - 6; }
// first global row and row count of stage k (k = N-1: the terminal rows)
KHD long long stage_row0(int N, int k) { return k == N - 1 ? 24 : 48 + (long long)ROWS_INT * k; }
KHD int stage_nrow(int N, int k) { return k == N - 1 ? 24 : k == N - 2 ? ROWS_LAST : ROWS_INT; }

// Device or host tables of the plan (make_kino_step_plan).  Stage k's terms are sorted by target; a segment is the run of
// terms of one target, summed in table order by one thread.
struct StepTables {
  int N;
  long long nx, m;
  const int *mstage, *mtgt, *mbeg, *mterm;  // M: [K+2] segment ranges, [nseg] target i*60+j (i >= j), [nseg+1], (a, b, lrow)
  const int *qstage, *qtgt, *qbeg, *qterm;  // q: same, (a, lrow): lrow < 0 -> grad_f[a]
  const int *dstage, *dterm;                // dynamics: [K+1] ranges, (jac pos, G index st*60 + scol)
  const int *rptr, *rent;                   // rows: [m+1], (jac pos, col) -- J by rows, for ds
};

// strided per-scenario vectors (element i at p[i * s])
struct SV {
  const double* p;
  long long s;
  KHD double operator[](long long i) const { return p[i * s]; }
};
struct MV {
  double* p;
  long long s;
  KHD double& operator[](long long i) const { return p[i * s]; }
};

// The iterate of one scenario.  `In` supplies jac(i), hess(i), gf(i) (the instrumented host build counts them).
struct StepPoint {
  SV g, s, y, zL, zU, lbg, ubg;
  double mu;
};

// sigma and yhat = sigma (g - s) + mu / (ubg - s) - mu / (s - lbg) of the stage's rows (0 on equality and free rows)
KHD void row_barrier(const StepPoint& it, long long i, double& sg, double& yh) {
  sg = 0.0; yh = 0.0;
  if (step_is_eq(i)) return;
  const double lo = it.lbg[i], up = it.ubg[i], s = it.s[i];
  if (lo > -HUGE_VAL) {
    const double d = s - lo;
    sg += it.zL[i] / d;
    yh -= it.mu / d;
  }
  if (up < HUGE_VAL) {
    const double d = up - s;
    sg += it.zU[i] / d;
    yh += it.mu / d;
  }
  yh += sg * (it.g[i] - s);
}

// Shared work arrays of one scenario (60 x 60 stage matrix and the rest: STEP_SMEM doubles).
constexpr int STEP_SMEM = SW * SW + 12 * SW + 24 * SW + 24 * 24 + 24 + SW + 2 * ROWS_INT + 24 + 24 + SU + 8;
struct StepShared {
  double *M, *Gz, *T, *P, *pv, *q, *sg, *yh, *t, *xi, *u, *red;
  KHD explicit StepShared(double* b)
      : M(b), Gz(M + SW * SW), T(Gz + 12 * SW), P(T + 24 * SW), pv(P + 24 * 24), q(pv + 24), sg(q + SW), yh(sg + ROWS_INT),
        t(yh + ROWS_INT), xi(t + 24), u(xi + 24), red(u + SU) {}
};
// factors of one stage in scratch: L (36 x 36 lower), Y (36 x 24), yv (36), Gz (12 x 60), r (12), P (24 x 24), p (24)
constexpr int STEP_STAGE = SU * SU + SU * SXI + SU + 12 * SW + 12 + 24 * 24 + 24;

// Assemble stage k: M (lower triangle) and q from the plan, Gz and r from the dynamics rows, and dw on the diagonal.
template <class In>
KHD void assemble_stage(const StepTables& tb, int k, const In& in, const StepPoint& it, double dw, StepShared& sh,
                        Team tm) {
  const int N = tb.N, K = N - 1;
  const long long row0 = stage_row0(N, k);
  const int nrow = stage_nrow(N, k);
  for (int i = tm.tid; i < SW * SW; i += tm.nt) sh.M[i] = 0.0;
  for (int i = tm.tid; i < 12 * SW; i += tm.nt) sh.Gz[i] = 0.0;
  for (int i = tm.tid; i < SW; i += tm.nt) sh.q[i] = 0.0;
  for (int i = tm.tid; i < nrow; i += tm.nt) row_barrier(it, row0 + i, sh.sg[i], sh.yh[i]);
  team_sync();
  for (int sgm = tb.mstage[k] + tm.tid; sgm < tb.mstage[k + 1]; sgm += tm.nt) {
    double acc = 0.0;
    for (int e = tb.mbeg[sgm]; e < tb.mbeg[sgm + 1]; e++) {
      const int a = tb.mterm[3 * e], b = tb.mterm[3 * e + 1], lr = tb.mterm[3 * e + 2];
      acc += lr < 0 ? in.hess(a) : sh.sg[lr] * (in.jac(a) * in.jac(b));
    }
    sh.M[tb.mtgt[sgm]] = acc;
  }
  for (int sgm = tb.qstage[k] + tm.tid; sgm < tb.qstage[k + 1]; sgm += tm.nt) {
    double acc = 0.0;
    for (int e = tb.qbeg[sgm]; e < tb.qbeg[sgm + 1]; e++) {
      const int a = tb.qterm[2 * e], lr = tb.qterm[2 * e + 1];
      acc += lr < 0 ? in.gf(a) : sh.yh[lr] * in.jac(a);
    }
    sh.q[tb.qtgt[sgm]] = acc;
  }
  if (k < K) {
    for (int e = tb.dstage[k] + tm.tid; e < tb.dstage[k + 1]; e += tm.nt) sh.Gz[tb.dterm[2 * e + 1]] = -in.jac(tb.dterm[2 * e]);
  }
  team_sync();
  const int nd = k == K ? 12 : 48;
  for (int i = tm.tid; i < nd; i += tm.nt) sh.M[i * SW + i] += dw;
  if (k == K - 1)
    for (int i = tm.tid; i < 12; i += tm.nt) sh.M[(48 + i) * SW + 48 + i] = 1.0;  // (no c_{N-1}: decoupled identity)
  team_sync();
}

// Backward step of stage k < N-1 with P_{k+1}, p_{k+1} in sh.P / sh.pv and the dynamics defect r in sh.t: forms
// Mh = M + A' P A, qh = q + A' (P b + p), factors its control block and leaves P_k, p_k in sh.P / sh.pv.  Returns false
// (uniformly over the team) when a pivot is <= 1e-14.
KHD bool riccati_stage(StepShared& sh, const double* r, double* Lout, double* Yout, double* yvout, Team tm) {
  double* M = sh.M;
  // T = [Pxx; Pcx] Gz (24 x 60), t = P (r, 0) + p
  for (int e = tm.tid; e < 24 * SW; e += tm.nt) {
    const int l = e / SW, j = e % SW;
    double acc = 0.0;
    for (int i = 0; i < 12; i++) acc += sh.P[l * 24 + i] * sh.Gz[i * SW + j];
    sh.T[e] = acc;
  }
  for (int i = tm.tid; i < 24; i += tm.nt) {
    double acc = sh.pv[i];
    for (int l = 0; l < 12; l++) acc += sh.P[i * 24 + l] * r[l];
    sh.t[i] = acc;
  }
  team_sync();
  for (int e = tm.tid; e < SW * SW; e += tm.nt) {
    const int i = e / SW, j = e % SW;
    if (j > i) continue;
    double acc = 0.0;
    for (int l = 0; l < 12; l++) acc += sh.Gz[l * SW + i] * sh.T[l * SW + j];
    if (j >= 48) acc += sh.T[(12 + j - 48) * SW + i];
    if (i >= 48) acc += sh.T[(12 + i - 48) * SW + j];
    if (i >= 48 && j >= 48) acc += sh.P[(12 + i - 48) * 24 + 12 + j - 48];
    M[e] += acc;
  }
  for (int j = tm.tid; j < SW; j += tm.nt) {
    double acc = sh.q[j];
    for (int l = 0; l < 12; l++) acc += sh.Gz[l * SW + j] * sh.t[l];
    if (j >= 48) acc += sh.t[12 + j - 48];
    sh.q[j] = acc;
  }
  // Cholesky of the control block M[24.., 24..] in place (right-looking)
  double* A = M + 24 * SW + 24;
  for (int j = 0; j < SU; j++) {
    team_sync();
    const double d = A[j * SW + j];
    if (!(d > 1e-14)) {
      team_sync();  // (every thread has read the pivot before the next trial overwrites M)
      return false;
    }
    const double sq = sqrt(d);
    team_sync();
    for (int i = j + 1 + tm.tid; i < SU; i += tm.nt) A[i * SW + j] /= sq;
    if (tm.tid == 0) A[j * SW + j] = sq;
    team_sync();
    const int n = SU - j - 1;
    for (int e = tm.tid; e < n * n; e += tm.nt) {
      const int i = j + 1 + e / n, l = j + 1 + e % n;
      if (l <= i) A[i * SW + l] -= A[i * SW + j] * A[l * SW + j];
    }
  }
  team_sync();
  // Y = L^-1 M_u,xi (36 x 24) and yv = L^-1 qh_u, one column per thread, in place
  for (int c = tm.tid; c <= SXI; c += tm.nt) {
    for (int i = 0; i < SU; i++) {
      double v = c < SXI ? M[(24 + i) * SW + c] : sh.q[24 + i];
      for (int l = 0; l < i; l++) v -= A[i * SW + l] * (c < SXI ? M[(24 + l) * SW + c] : sh.q[24 + l]);
      v /= A[i * SW + i];
      if (c < SXI) M[(24 + i) * SW + c] = v;
      else sh.q[24 + i] = v;
    }
  }
  team_sync();
  // P_k = M_xi,xi - Y'Y, p_k = qh_xi - Y' yv
  for (int e = tm.tid; e < 24 * 24; e += tm.nt) {
    const int i = e / 24, j = e % 24;
    if (j > i) continue;
    double v = M[i * SW + j];
    for (int l = 0; l < SU; l++) v -= M[(24 + l) * SW + i] * M[(24 + l) * SW + j];
    sh.P[i * 24 + j] = v;
    sh.P[j * 24 + i] = v;
  }
  for (int i = tm.tid; i < 24; i += tm.nt) {
    double v = sh.q[i];
    for (int l = 0; l < SU; l++) v -= M[(24 + l) * SW + i] * sh.q[24 + l];
    sh.pv[i] = v;
  }
  for (int e = tm.tid; e < SU * SU; e += tm.nt) Lout[e] = A[(e / SU) * SW + e % SU];
  for (int e = tm.tid; e < SU * SXI; e += tm.nt) Yout[e] = M[(24 + e / SXI) * SW + e % SXI];
  for (int i = tm.tid; i < SU; i += tm.nt) yvout[i] = sh.q[24 + i];
  team_sync();
  return true;
}

// Backward sweep with regularisation dw: the factors of every stage to scr (STEP_STAGE doubles per stage).  false: wrong
// inertia.
template <class In>
KHD bool step_factor(const StepTables& tb, const In& in, const StepPoint& it, double dw, StepShared& sh, double* scr,
                     Team tm) {
  const int N = tb.N, K = N - 1;
  // terminal block
  assemble_stage(tb, K, in, it, dw, sh, tm);
  for (int e = tm.tid; e < 24 * 24; e += tm.nt) {
    const int i = e / 24, j = e % 24;
    const double v = sh.M[(i > j ? i : j) * SW + (i > j ? j : i)];
    sh.P[e] = v;
  }
  for (int i = tm.tid; i < 24; i += tm.nt) sh.pv[i] = sh.q[i];
  team_sync();
  for (int k = K - 1; k >= 0; k--) {
    double* st = scr + (size_t)(k + 1) * STEP_STAGE;  // P_{k+1}, p_{k+1} of this sweep
    double* Ps = st + SU * SU + SU * SXI + SU + 12 * SW + 12;
    for (int e = tm.tid; e < 24 * 24; e += tm.nt) Ps[e] = sh.P[e];
    for (int i = tm.tid; i < 24; i += tm.nt) Ps[576 + i] = sh.pv[i];
    assemble_stage(tb, k, in, it, dw, sh, tm);
    double* sk = scr + (size_t)k * STEP_STAGE;
    double* r = sk + SU * SU + SU * SXI + SU + 12 * SW;
    const long long row0 = stage_row0(N, k);
    for (int rho = tm.tid; rho < 12; rho += tm.nt) r[dynrow_state(rho)] = -it.g[row0 + rho];
    for (int e = tm.tid; e < 12 * SW; e += tm.nt) sk[SU * SU + SU * SXI + SU + e] = sh.Gz[e];
    team_sync();
    if (!riccati_stage(sh, r, sk, sk + SU * SU, sk + SU * SU + SU * SXI, tm)) return false;
  }
  double* Ps = scr + SU * SU + SU * SXI + SU + 12 * SW + 12;  // P_0, p_0
  for (int e = tm.tid; e < 24 * 24; e += tm.nt) Ps[e] = sh.P[e];
  for (int i = tm.tid; i < 24; i += tm.nt) Ps[576 + i] = sh.pv[i];
  team_sync();
  return true;
}

struct StepOut {
  MV dx, ds, dy, dzL, dzU;
};

// Forward sweep: dx, and dy of the equality rows (costates); then ds, dy, dzL, dzU of every inequality row and the
// fraction-to-boundary step lengths (tau > 0).
template <class In>
KHD void step_solve(const StepTables& tb, const In& in, const StepPoint& it, const double* scr, StepShared& sh,
                    const StepOut& o, double tau, double* a_pr, double* a_du, Team tm) {
  const int N = tb.N, K = N - 1;
  const long long cU = 24LL * N - 12;
  for (int i = tm.tid; i < 24; i += tm.nt) sh.xi[i] = -(it.g[i] - it.lbg[i]);
  team_sync();
  {
    const double* P0 = scr + SU * SU + SU * SXI + SU + 12 * SW + 12;
    for (int i = tm.tid; i < 24; i += tm.nt) {
      double v = P0[576 + i];
      for (int l = 0; l < 24; l++) v += P0[i * 24 + l] * sh.xi[l];
      o.dy[i] = -v - it.y[i];
    }
  }
  for (int k = 0; k < K; k++) {
    const double* sk = scr + (size_t)k * STEP_STAGE;
    const double *L = sk, *Y = sk + SU * SU, *yv = Y + SU * SXI, *Gz = yv + SU, *r = Gz + 12 * SW;
    // u = -L^-T (yv + Y xi): the right-hand side in sh.t / sh.u, then a column sweep of L'
    for (int i = tm.tid; i < SU; i += tm.nt) {
      double v = yv[i];
      for (int l = 0; l < SXI; l++) v += Y[i * SXI + l] * sh.xi[l];
      sh.u[i] = -v;
    }
    for (int i = SU - 1; i >= 0; i--) {
      team_sync();
      const double ui = sh.u[i] / L[i * SU + i];
      team_sync();
      for (int l = tm.tid; l < i; l += tm.nt) sh.u[l] -= L[i * SU + l] * ui;
      if (tm.tid == 0) sh.u[i] = ui;
    }
    team_sync();
    for (int i = tm.tid; i < 12; i += tm.nt) {
      o.dx[12LL * k + i] = sh.xi[i];
      o.dx[cU + 24LL * k + i] = sh.xi[12 + i];
      o.dx[12LL * N + 12LL * k + i] = sh.u[i];
      o.dx[cU + 24LL * k + 12 + i] = sh.u[12 + i];
    }
    // xi_{k+1} = (Gz (xi, u) + r, c_{k+1})
    for (int i = tm.tid; i < 24; i += tm.nt) {
      double v;
      if (i < 12) {
        v = r[i];
        for (int j = 0; j < SXI; j++) v += Gz[i * SW + j] * sh.xi[j];
        for (int j = 0; j < SU; j++) v += Gz[i * SW + 24 + j] * sh.u[j];
      } else {
        v = k == K - 1 ? 0.0 : sh.u[24 + i - 12];
      }
      sh.t[i] = v;
    }
    team_sync();
    for (int i = tm.tid; i < 24; i += tm.nt) sh.xi[i] = sh.t[i];
    // costates: dynamics row rho of knot k, y + dy = -(P_{k+1} xi_{k+1} + p_{k+1})[state of rho]
    const double* Pn = scr + (size_t)(k + 1) * STEP_STAGE + SU * SU + SU * SXI + SU + 12 * SW + 12;
    const long long row0 = stage_row0(N, k);
    for (int rho = tm.tid; rho < 12; rho += tm.nt) {
      const int st = dynrow_state(rho);
      double v = Pn[576 + st];
      for (int l = 0; l < 24; l++) v += Pn[st * 24 + l] * sh.t[l];
      o.dy[row0 + rho] = -v - it.y[row0 + rho];
    }
    team_sync();
  }
  for (int i = tm.tid; i < 12; i += tm.nt) o.dx[12LL * K + i] = sh.xi[i];
  team_sync();
  // recovery, parallel over rows
  double apr = 1.0, adu = 1.0;
  for (long long i = tm.tid; i < tb.m; i += tm.nt) {
    if (step_is_eq(i)) {
      o.ds[i] = 0.0; o.dzL[i] = 0.0; o.dzU[i] = 0.0;
      continue;
    }
    const double s = it.s[i], lo = it.lbg[i], up = it.ubg[i];
    double ds = it.g[i] - s;
    for (int e = tb.rptr[i]; e < tb.rptr[i + 1]; e++) ds += in.jac(tb.rent[2 * e]) * o.dx[tb.rent[2 * e + 1]];
    double sg = 0.0, yn = 0.0, dzl = 0.0, dzu = 0.0;
    if (lo > -HUGE_VAL) {
      const double d = s - lo, z = it.zL[i];
      sg += z / d;
      yn -= it.mu / d;
      dzl = it.mu / d - z - z / d * ds;
      if (ds < 0) apr = fmin(apr, -tau * (s - lo) / ds);
      if (dzl < 0) adu = fmin(adu, -tau * z / dzl);
    }
    if (up < HUGE_VAL) {
      const double d = up - s, z = it.zU[i];
      sg += z / d;
      yn += it.mu / d;
      dzu = it.mu / d - z + z / d * ds;
      if (ds > 0) apr = fmin(apr, tau * (up - s) / ds);
      if (dzu < 0) adu = fmin(adu, -tau * z / dzu);
    }
    yn += sg * ds;
    o.ds[i] = ds; o.dzL[i] = dzl; o.dzU[i] = dzu;
    o.dy[i] = yn - it.y[i];
  }
  *a_pr = apr;
  *a_du = adu;
}

// Is the iterate interior on every finite bound of an inequality row (strictly, and no NaN)?  Per thread.
KHD bool step_interior(const StepPoint& it, long long m, Team tm) {
  bool ok = true;
  for (long long i = tm.tid; i < m; i += tm.nt) {
    if (step_is_eq(i)) continue;
    const double s = it.s[i], lo = it.lbg[i], up = it.ubg[i];
    if (lo > -HUGE_VAL) ok = ok && (s - lo > 0.0) && (it.zL[i] > 0.0);
    if (up < HUGE_VAL) ok = ok && (up - s > 0.0) && (it.zU[i] > 0.0);
  }
  return ok;
}

// IPOPT's inertia-correction schedule (oracle/ip_ref.c, ip_solve_ws): the first trial value from the previous
// iteration's dw_last, the next one after a failed factorisation.  `tries` counts the failures so far.
KHD double dw_first(double dw_last) {
  if (dw_last > 0) {
    const double d = dw_last / 3.0;
    return d < 1e-7 ? 0.0 : d;
  }
  return 0.0;
}
KHD double dw_next(double dw, double dw_last, int tries) {
  if (dw == 0) return dw_last == 0 ? 1e-4 : fmax(1e-20, dw_last / 3.0);
  return dw * ((dw_last == 0 && tries < 8) ? 100.0 : 8.0);
}

// ---------------------------------------------------------------- host plan (once per N)
struct KinoStepPlan {
  int N = 0;
  long long nx = 0, m = 0;
  std::vector<int> mstage, mtgt, mbeg, mterm, qstage, qtgt, qbeg, qterm, dstage, dterm, rptr, rent;
  std::vector<int> jrole;  // per Jacobian entry: 0 boundary identity, 1 X_{k+1} identity, 2 dynamics (G), 3 inequality row
  std::string err;
};

// stages holding column col: up to two (stage, stage column); returns the count
inline int step_col_stages(int N, long long col, int st[2], int sc[2]) {
  const long long cJ = 12LL * N, cU = 24LL * N - 12;
  if (col < cJ) { st[0] = (int)(col / 12); sc[0] = (int)(col % 12); return 1; }  // X_j (j = N-1: the terminal stage)
  if (col < cU) { st[0] = (int)((col - cJ) / 12); sc[0] = 24 + (int)((col - cJ) % 12); return 1; }
  const int j = (int)((col - cU) / 24), i = (int)((col - cU) % 24);
  if (i >= 12) { st[0] = j; sc[0] = 36 + i - 12; return 1; }
  st[0] = j; sc[0] = 12 + i;  // c_j: state of stage j, control of stage j - 1
  if (j >= 1) { st[1] = j - 1; sc[1] = 48 + i; return 2; }
  return 1;
}
inline int step_col_in(int N, long long col, int stage) {  // stage column of col in stage, or -1
  int st[2], sc[2];
  const int n = step_col_stages(N, col, st, sc);
  for (int a = 0; a < n; a++)
    if (st[a] == stage) return sc[a];
  return -1;
}

// From the CCS patterns of J (colind, row) and of the upper triangle of W: every Jacobian entry to its stage, row and
// stage column, every Hessian entry and every grad_f column to exactly one stage matrix.  err is set (and the tables are
// unusable) for an entry outside every stage.
inline KinoStepPlan make_kino_step_plan(int N, const long long* jcol, const long long* jrow, const long long* hcol,
                                        const long long* hrow) {
  KinoStepPlan pl;
  pl.N = N;
  const int K = N - 1, S = K + 1;
  pl.nx = 12LL * N + 36LL * (N - 1);
  pl.m = 48 + (long long)ROWS_INT * (N - 2) + ROWS_LAST;
  const long long nx = pl.nx, m = pl.m, nnzJ = jcol[nx];
  struct MT { int stage, tgt, a, b, lr; };
  struct QT { int stage, tgt, a, lr; };
  std::vector<MT> mt;
  std::vector<QT> qt;
  std::vector<std::vector<std::pair<int, int>>> rows((size_t)m);  // per row: (jac pos, stage column)
  std::vector<std::pair<int, int>> dyn;                           // (stage, index into dterm)
  std::vector<int> dt;
  pl.jrole.assign((size_t)nnzJ, -1);
  std::vector<std::vector<std::pair<int, long long>>> byrow((size_t)m);
  auto fail = [&](const std::string& e) { pl.err = "kino step plan: " + e; return pl; };
  for (long long c = 0; c < nx; c++)
    for (long long e = jcol[c]; e < jcol[c + 1]; e++) {
      const long long r = jrow[e];
      if (r < 0 || r >= m) return fail("Jacobian row out of range");
      byrow[(size_t)r].push_back({(int)e, c});
      if (r < 24) {  // x_0 - q_init, c_0 - c_init
        if (c != (r < 12 ? r : 24LL * N - 12 + (r - 12))) return fail("boundary row " + std::to_string(r) + " off its column");
        pl.jrole[(size_t)e] = 0;
        continue;
      }
      const int k = r < 48 ? K : (int)((r - 48) / ROWS_INT);
      const int lr = (int)(r - stage_row0(N, k));
      if (k < K && lr < 12) {  // dynamics row
        const int st = dynrow_state(lr);
        if (c == 12LL * (k + 1) + st) { pl.jrole[(size_t)e] = 1; continue; }
        const int sc = step_col_in(N, c, k);
        if (sc < 0 || (sc >= 24 && sc < 36) || sc >= 48)
          return fail("dynamics entry (" + std::to_string(r) + ", " + std::to_string(c) + ") outside its stage");
        pl.jrole[(size_t)e] = 2;
        dyn.push_back({k, (int)dt.size() / 2});
        dt.push_back((int)e);
        dt.push_back(st * SW + sc);
        continue;
      }
      const int sc = step_col_in(N, c, k);
      if (sc < 0) return fail("entry (" + std::to_string(r) + ", " + std::to_string(c) + ") outside its stage");
      pl.jrole[(size_t)e] = 3;
      rows[(size_t)r].push_back({(int)e, sc});
    }
  for (long long r = 24; r < m; r++) {
    if (step_is_eq(r)) continue;
    const int k = r < 48 ? K : (int)((r - 48) / ROWS_INT);
    const int lr = (int)(r - stage_row0(N, k));
    const auto& R = rows[(size_t)r];
    for (size_t a = 0; a < R.size(); a++) {
      qt.push_back({k, R[a].second, R[a].first, lr});
      for (size_t b = 0; b <= a; b++) {
        const int i = std::max(R[a].second, R[b].second), j = std::min(R[a].second, R[b].second);
        mt.push_back({k, i * SW + j, R[a].first, R[b].first, lr});
      }
    }
  }
  for (long long c = 0; c < nx; c++)
    for (long long e = hcol[c]; e < hcol[c + 1]; e++) {
      const long long r = hrow[e];
      int sa[2], ca[2];
      const int na = step_col_stages(N, c, sa, ca);
      int best = -1, i = 0, j = 0;
      for (int a = 0; a < na; a++) {
        const int sr = step_col_in(N, r, sa[a]);
        if (sr >= 0 && sa[a] > best) { best = sa[a]; i = std::max(ca[a], sr); j = std::min(ca[a], sr); }
      }
      if (best < 0) return fail("Hessian entry (" + std::to_string(r) + ", " + std::to_string(c) + ") outside every stage");
      mt.push_back({best, i * SW + j, (int)e, 0, -1});
    }
  for (long long c = 0; c < nx; c++) {
    int st[2], sc[2];
    step_col_stages(N, c, st, sc);
    qt.push_back({st[0], sc[0], (int)c, -1});  // (the later stage: c_j to stage j, as the Hessian)
  }
  // a stage matrix entry must come from one stage only: sort by (stage, target), keeping table order within a target
  std::stable_sort(mt.begin(), mt.end(), [](const MT& x, const MT& y) { return x.stage != y.stage ? x.stage < y.stage : x.tgt < y.tgt; });
  std::stable_sort(qt.begin(), qt.end(), [](const QT& x, const QT& y) { return x.stage != y.stage ? x.stage < y.stage : x.tgt < y.tgt; });
  pl.mstage.assign(S + 1, 0);
  pl.qstage.assign(S + 1, 0);
  for (size_t e = 0; e < mt.size(); e++) {
    if (e == 0 || mt[e].stage != mt[e - 1].stage || mt[e].tgt != mt[e - 1].tgt) {
      pl.mtgt.push_back(mt[e].tgt);
      pl.mbeg.push_back((int)e);
      pl.mstage[mt[e].stage + 1] = (int)pl.mtgt.size();
    }
    pl.mterm.push_back(mt[e].a); pl.mterm.push_back(mt[e].b); pl.mterm.push_back(mt[e].lr);
  }
  pl.mbeg.push_back((int)mt.size());
  for (size_t e = 0; e < qt.size(); e++) {
    if (e == 0 || qt[e].stage != qt[e - 1].stage || qt[e].tgt != qt[e - 1].tgt) {
      pl.qtgt.push_back(qt[e].tgt);
      pl.qbeg.push_back((int)e);
      pl.qstage[qt[e].stage + 1] = (int)pl.qtgt.size();
    }
    pl.qterm.push_back(qt[e].a); pl.qterm.push_back(qt[e].lr);
  }
  pl.qbeg.push_back((int)qt.size());
  for (int s = 1; s <= S; s++) {  // (stages without terms)
    pl.mstage[s] = std::max(pl.mstage[s], pl.mstage[s - 1]);
    pl.qstage[s] = std::max(pl.qstage[s], pl.qstage[s - 1]);
  }
  pl.dstage.assign(K + 1, 0);
  {
    std::vector<int> order(dyn.size());
    for (size_t i = 0; i < dyn.size(); i++) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return dyn[a].first < dyn[b].first; });
    for (int o : order) {
      pl.dterm.push_back(dt[2 * dyn[o].second]);
      pl.dterm.push_back(dt[2 * dyn[o].second + 1]);
      pl.dstage[dyn[o].first + 1] += 1;
    }
    for (int k = 0; k < K; k++) pl.dstage[k + 1] += pl.dstage[k];
  }
  pl.rptr.assign((size_t)m + 1, 0);
  for (long long r = 0; r < m; r++) {
    pl.rptr[(size_t)r + 1] = pl.rptr[(size_t)r] + (int)byrow[(size_t)r].size();
    for (auto& p : byrow[(size_t)r]) { pl.rent.push_back(p.first); pl.rent.push_back((int)p.second); }
  }
  return pl;
}

}  // namespace kino
}  // namespace srb
