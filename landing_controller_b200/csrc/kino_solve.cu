// kino_solve.cu -- batched interior-point solve of the kino-dynamic ("full-body") landing NLP (include/landing_b200.h:
// landing_kino_solve_batch).  The method is the primal-dual filter line search of oracle/ip_ref.c (ip_solve_ws), with
// its constants and deviations (DESIGN.md 3, 3.2); the evaluations and the Newton step are the library's existing
// launchers (launch_kino, launch_kino_cost, launch_kino_hess, launch_kino_grad, launch_kino_kkt, launch_kino_step).
//
// The loop runs on the host over device-resident SoA state ([rows][B_run], one column per running scenario).  One outer
// round: grad_x of the Lagrangian and the final measures at x; k_ks_measure (E0, termination, the barrier update); a
// stable compaction of the running scenarios to the front when some finished (their results go to the caller's
// buffers); the Jacobian, cost gradient and Hessian of the running ones, then the step; k_ks_ftb
// (fraction to the boundary, merit, dphi); line-search rounds over the scenarios still searching (k_ks_trial, g and f
// at the trial points, k_ks_filter); k_ks_accept (accept or re-centre).  Every bookkeeping kernel is one thread per
// scenario summing its rows in a fixed order, so a scenario's arithmetic does not depend on its slot or companions.
// The host reads back one count per outer round (running) and one per line-search round (searching).
#include <string>

#include "kernels.cuh"

namespace srb {
namespace {

constexpr int MAXF = 64;  // filter entries per scenario (oracle/ip_ref.c MAXFILTER)
constexpr int NT = 128;

// persistent state of the running scenarios, stride n (double-buffered: compaction gathers into the other copy)
struct PS {
  long long n;
  double *x, *s, *y, *zL, *zU, *g, *lb, *ub, *lbo, *ubo, *f, *mu, *dwl, *th0, *fth, *fph;
  int *status, *iters, *rest, *tiny, *nfilt, *orig;
};
// quantities of the current round, stride n
struct RS {
  long long n;
  double *jac, *hess, *gf, *gl, *dx, *ds, *dy, *dzL, *dzU, *dw, *apr, *adu, *phi, *th, *dphi, *alpha, *fv, *fd, *fc;
  int *nf, *sst, *ls, *srch, *acc, *ftype;
};
// trial points of the scenarios still searching, stride n
struct TS {
  long long n;
  double *xt, *gt, *ft;
};

struct Dims {
  int N;
  long long nx, m, nnzJ, nnzH;
  long long pd() const { return nx + 9 * m + 4 + 2 * MAXF; }
  long long rd() const { return nnzJ + nnzH + 3 * nx + 4 * m + 10; }
  long long td() const { return nx + m + 1; }
};
constexpr long long PI_ROWS = 6, RI_ROWS = 6;

struct Take {
  double* d;
  long long n;
  double* operator()(long long rows) { double* r = d; d += rows * n; return r; }
};
struct TakeI {
  int* d;
  long long n;
  int* operator()(long long rows) { int* r = d; d += rows * n; return r; }
};
PS make_ps(double* d, int* iv, long long n, const Dims& D) {
  PS p;
  p.n = n;
  Take t{d, n};
  p.x = t(D.nx); p.s = t(D.m); p.y = t(D.m); p.zL = t(D.m); p.zU = t(D.m); p.g = t(D.m); p.lb = t(D.m); p.ub = t(D.m);
  p.lbo = t(D.m); p.ubo = t(D.m); p.f = t(1); p.mu = t(1); p.dwl = t(1); p.th0 = t(1); p.fth = t(MAXF); p.fph = t(MAXF);
  TakeI ti{iv, n};
  p.status = ti(1); p.iters = ti(1); p.rest = ti(1); p.tiny = ti(1); p.nfilt = ti(1); p.orig = ti(1);
  return p;
}
RS make_rs(double* d, int* iv, long long n, const Dims& D) {
  RS r;
  r.n = n;
  Take t{d, n};
  r.jac = t(D.nnzJ); r.hess = t(D.nnzH); r.gf = t(D.nx); r.gl = t(D.nx); r.dx = t(D.nx);
  r.ds = t(D.m); r.dy = t(D.m); r.dzL = t(D.m); r.dzU = t(D.m);
  r.dw = t(1); r.apr = t(1); r.adu = t(1); r.phi = t(1); r.th = t(1); r.dphi = t(1); r.alpha = t(1);
  r.fv = t(1); r.fd = t(1); r.fc = t(1);
  TakeI ti{iv, n};
  r.nf = ti(1); r.sst = ti(1); r.ls = ti(1); r.srch = ti(1); r.acc = ti(1); r.ftype = ti(1);
  return r;
}
TS make_ts(double* d, long long n, const Dims& D) {
  TS t;
  t.n = n;
  Take k{d, n};
  t.xt = k(D.nx); t.gt = k(D.m); t.ft = k(1);
  return t;
}

struct Opt {  // landing_options, as the kernels use them
  int max_iter, jam_iters, max_restarts;
  double tol, cvt, dit, cit, mu_init, bound_push, bound_frac, brf, jam_alpha, restart_mu;
};

__device__ __forceinline__ bool finite_lo(double v) { return v > -HUGE_VAL; }
__device__ __forceinline__ bool finite_up(double v) { return v < HUGE_VAL; }

// oracle/ip_ref.c init_slacks: slacks pushed inside the (relaxed) bounds at the current g, mu-based bound multipliers,
// y = zU - zL on inequality rows, 0 on equality rows
__device__ void init_slacks(const PS& p, long long b, long long m, const Opt& o, double mu) {
  const long long n = p.n;
  for (long long i = 0; i < m; i++) {
    const long long e = i * n + b;
    double s = 0.0, zl = 0.0, zu = 0.0;
    if (!kino::step_is_eq(i)) {
      const double l = p.lb[e], u = p.ub[e];
      s = p.g[e];
      if (finite_lo(l) && finite_up(u)) {
        const double pL = fmin(o.bound_push * fmax(1.0, fabs(l)), o.bound_frac * (u - l));
        const double pU = fmin(o.bound_push * fmax(1.0, fabs(u)), o.bound_frac * (u - l));
        s = fmin(fmax(s, l + pL), u - pU);
      } else if (finite_lo(l)) {
        s = fmax(s, l + o.bound_push * fmax(1.0, fabs(l)));
      } else {
        s = fmin(s, u - o.bound_push * fmax(1.0, fabs(u)));
      }
      if (finite_lo(l)) zl = mu / (s - l);
      if (finite_up(u)) zu = mu / (u - s);
    }
    p.s[e] = s; p.zL[e] = zl; p.zU[e] = zu;
    p.y[e] = zu - zl;
  }
}

// caller's AoS initial guess -> state
__global__ void k_ks_load(PS p, const double* x0, long long nx) {
  const long long b = (long long)blockIdx.x * NT + threadIdx.x;
  if (b >= p.n) return;
  for (long long i = blockIdx.y; i < nx; i += gridDim.y) p.x[i * p.n + b] = x0[b * nx + i];
}

// relaxed bounds on the inequality rows, slacks and multipliers, scalars (the start of ip_solve_ws)
__global__ void k_ks_init(PS p, long long m, Opt o) {
  const long long b = (long long)blockIdx.x * NT + threadIdx.x;
  if (b >= p.n) return;
  const long long n = p.n;
  for (long long i = 0; i < m; i++) {
    const long long e = i * n + b;
    double l = p.lbo[e], u = p.ubo[e];
    if (!kino::step_is_eq(i)) {
      if (isfinite(l)) l -= o.brf * fmax(1.0, fabs(l));
      if (isfinite(u)) u += o.brf * fmax(1.0, fabs(u));
    }
    p.lb[e] = l; p.ub[e] = u;
  }
  init_slacks(p, b, m, o, o.mu_init);
  p.mu[b] = o.mu_init; p.dwl[b] = 0.0; p.th0[b] = -1.0;
  p.status[b] = LANDING_ST_RUNNING; p.iters[b] = 0; p.rest[b] = 0; p.tiny[b] = 0; p.nfilt[b] = 0; p.orig[b] = (int)b;
}

// IPOPT's scaled optimality error E0 (ip_ref.c assemble / ip_solve_ws), the termination test, the monotone barrier
// update with the filter reset.  A NaN in any quantity the measures read gives LANDING_ST_NAN.
__global__ void k_ks_measure(PS p, RS r, long long m, long long nx, Opt o) {
  const long long b = (long long)blockIdx.x * NT + threadIdx.x;
  if (b >= p.n || p.status[b] != LANDING_ST_RUNNING) return;
  const long long n = p.n;
  double mu = p.mu[b];
  double dual = 0, prim = 0, c0 = 0, cmu = 0, ys = 0, zs = 0, viol = 0;
  long long nb = 0;
  bool nan = isnan(p.f[b]);
  for (long long i = 0; i < m; i++) {
    const long long e = i * n + b;
    const double gi = p.g[e], yi = p.y[e], lo = p.lb[e], up = p.ub[e], lbo = p.lbo[e], ubo = p.ubo[e];
    nan = nan || isnan(gi) || isnan(yi) || isnan(lbo) || isnan(ubo);
    viol = fmax(viol, fmax(lbo - gi, gi - ubo));
    ys += fabs(yi);
    if (kino::step_is_eq(i)) {
      prim = fmax(prim, fabs(gi - lo));
      continue;
    }
    const double si = p.s[e];
    double rs = -yi;
    nan = nan || isnan(si);
    if (finite_lo(lo)) {
      const double d = si - lo, z = p.zL[e];
      nan = nan || isnan(z);
      rs -= z;
      c0 = fmax(c0, fabs(z * d));
      cmu = fmax(cmu, fabs(z * d - mu));
      zs += z;
      nb++;
    }
    if (finite_up(up)) {
      const double d = up - si, z = p.zU[e];
      nan = nan || isnan(z);
      rs += z;
      c0 = fmax(c0, fabs(z * d));
      cmu = fmax(cmu, fabs(z * d - mu));
      zs += z;
      nb++;
    }
    prim = fmax(prim, fabs(gi - si));
    dual = fmax(dual, fabs(rs));
  }
  for (long long j = 0; j < nx; j++) {
    const double v = r.gl[j * n + b];
    nan = nan || isnan(v);
    dual = fmax(dual, fabs(v));
  }
  const double s_max = 100.0;
  const double s_d = fmax(s_max, (ys + zs) / (double)(m + nb)) / s_max;
  const double s_c = fmax(s_max, zs / (double)(nb > 0 ? nb : 1)) / s_max;
  const double E0 = fmax(fmax(dual / s_d, prim), c0 / s_c);
  if (nan || !isfinite(E0) || !isfinite(p.f[b])) { p.status[b] = LANDING_ST_NAN; return; }
  if (E0 <= o.tol && dual <= o.dit && viol <= o.cvt && c0 <= o.cit) { p.status[b] = LANDING_ST_CONVERGED; return; }
  if (p.iters[b] == o.max_iter) { p.status[b] = LANDING_ST_MAX_ITER; return; }
  bool changed = false;
  for (;;) {
    const double Emu = fmax(fmax(dual / s_d, prim), cmu / s_c);
    if (!(Emu <= 10.0 * mu) || mu <= o.tol / 10.0 * 1.0000001) break;
    mu = fmax(o.tol / 10.0, fmin(0.2 * mu, pow(mu, 1.5)));
    changed = true;
    cmu = 0;
    for (long long i = 0; i < m; i++) {
      if (kino::step_is_eq(i)) continue;
      const long long e = i * n + b;
      const double si = p.s[e], lo = p.lb[e], up = p.ub[e];
      if (finite_lo(lo)) cmu = fmax(cmu, fabs(p.zL[e] * (si - lo) - mu));
      if (finite_up(up)) cmu = fmax(cmu, fabs(p.zU[e] * (up - si) - mu));
    }
  }
  if (changed) p.nfilt[b] = 0;
  p.mu[b] = mu;
}

// flags -> stable list of the indices with src[b] == want, and their count (one block)
constexpr int SCAN_NT = 1024;
__global__ void __launch_bounds__(SCAN_NT) k_ks_scan(const int* src, int want, long long n, int* map, int* count) {
  __shared__ int sh[SCAN_NT];
  const int t = threadIdx.x;
  const long long chunk = (n + SCAN_NT - 1) / SCAN_NT, lo = t * chunk, hi = lo + chunk < n ? lo + chunk : n;
  int c = 0;
  for (long long b = lo; b < hi; b++) c += src[b] == want;
  sh[t] = c;
  __syncthreads();
  for (int off = 1; off < SCAN_NT; off <<= 1) {  // inclusive scan
    const int v = t >= off ? sh[t - off] : 0;
    __syncthreads();
    sh[t] += v;
    __syncthreads();
  }
  int pos = sh[t] - c;
  for (long long b = lo; b < hi; b++)
    if (src[b] == want) map[pos++] = (int)b;
  if (t == SCAN_NT - 1) *count = sh[t];
}

struct Out {
  double *x_star, *f_star, *lam_g, *viol, *dual_inf, *compl_inf;
  int *status, *iters, *restarts;
};
// results of the scenarios that have finished, to the caller's (AoS) buffers at their original index
__global__ void k_ks_output(PS p, RS r, long long nx, long long m, Out o) {
  const long long b = (long long)blockIdx.x * NT + threadIdx.x;
  if (b >= p.n || p.status[b] == LANDING_ST_RUNNING) return;
  const long long ob = p.orig[b], n = p.n;
  for (long long i = blockIdx.y; i < nx + m; i += gridDim.y) {
    if (i < nx) o.x_star[ob * nx + i] = p.x[i * n + b];
    else if (o.lam_g) o.lam_g[ob * m + i - nx] = p.y[(i - nx) * n + b];
  }
  if (blockIdx.y == 0) {
    o.f_star[ob] = p.f[b];
    o.status[ob] = p.status[b];
    o.iters[ob] = p.iters[b];
    if (o.restarts) o.restarts[ob] = p.rest[b];
    if (o.viol) o.viol[ob] = r.fv[b];
    if (o.dual_inf) o.dual_inf[ob] = r.fd[b];
    if (o.compl_inf) o.compl_inf[ob] = r.fc[b];
  }
}

// stable gather of the running scenarios: dst[row][j] = src[row][map[j]]
template <class T>
__global__ void k_ks_gather(const T* src, long long no, T* dst, long long nn, long long rows, const int* map) {
  const long long j = (long long)blockIdx.x * NT + threadIdx.x;
  if (j >= nn) return;
  const long long b = map[j];
  for (long long i = blockIdx.y; i < rows; i += gridDim.y) dst[i * nn + j] = src[i * no + b];
}

// fraction to the boundary with the scenario's own tau, barrier merit phi, infeasibility theta and the directional
// derivative dphi at the current point (ip_ref.c ip_solve_ws after the step); the start of the line search
__global__ void k_ks_ftb(PS p, RS r, long long m, int N) {
  const long long b = (long long)blockIdx.x * NT + threadIdx.x;
  if (b >= p.n) return;
  r.srch[b] = 0;
  if (p.status[b] != LANDING_ST_RUNNING) return;
  if (r.sst[b] != 0) {  // no step: wrong inertia to the end of the schedule, or an iterate that is not interior
    p.status[b] = r.sst[b] == LANDING_ST_NOT_INTERIOR ? LANDING_ST_NAN : LANDING_ST_FACTOR_FAIL;
    return;
  }
  const long long n = p.n;
  p.dwl[b] = r.dw[b];
  const double mu = p.mu[b], tau = fmax(0.99, 1.0 - mu);
  double apr = 1.0, adu = 1.0, ph = p.f[b], th = 0.0, dphi = 0.0;
  for (int i = 0; i < 12; i++) {
    const long long c = 12LL * (N - 1) + i;
    dphi += r.gf[c * n + b] * r.dx[c * n + b];
  }
  for (long long i = 0; i < m; i++) {
    const long long e = i * n + b;
    const double gi = p.g[e], lo = p.lb[e], up = p.ub[e];
    if (kino::step_is_eq(i)) {
      th += fabs(gi - lo);
      continue;
    }
    const double si = p.s[e], ds = r.ds[e];
    th += fabs(gi - si);
    if (finite_lo(lo)) {
      const double d = si - lo, z = p.zL[e], dz = r.dzL[e];
      ph -= mu * log(d);
      dphi -= mu * ds / d;
      if (ds < 0) apr = fmin(apr, -tau * d / ds);
      if (dz < 0) adu = fmin(adu, -tau * z / dz);
    }
    if (finite_up(up)) {
      const double d = up - si, z = p.zU[e], dz = r.dzU[e];
      ph -= mu * log(d);
      dphi += mu * ds / d;
      if (ds > 0) apr = fmin(apr, tau * d / ds);
      if (dz < 0) adu = fmin(adu, -tau * z / dz);
    }
  }
  if (p.th0[b] < 0) p.th0[b] = th;
  r.apr[b] = apr; r.adu[b] = adu; r.phi[b] = ph; r.th[b] = th; r.dphi[b] = dphi;
  r.alpha[b] = apr; r.ls[b] = 0; r.acc[b] = 0; r.ftype[b] = 0;
  r.srch[b] = apr > 1e-12 * apr ? 1 : 0;
}

// trial points x + alpha dx of the scenarios still searching (map: their slots)
__global__ void k_ks_trial(PS p, RS r, TS t, long long nx, const int* map) {
  const long long j = (long long)blockIdx.x * NT + threadIdx.x;
  if (j >= t.n) return;
  const long long b = map[j], n = p.n;
  const double a = r.alpha[b];
  for (long long i = blockIdx.y; i < nx; i += gridDim.y) t.xt[i * t.n + j] = p.x[i * n + b] + a * r.dx[i * n + b];
}

// filter test of the trial point (ip_ref.c: filter with switching condition and Armijo test); the watchdog against
// jamming; an accepted trial is committed (x, g, f), a rejected one halves alpha
__global__ void k_ks_filter(PS p, RS r, TS t, long long nx, long long m, Opt o, const int* map) {
  const long long j = (long long)blockIdx.x * NT + threadIdx.x;
  if (j >= t.n) return;
  const long long b = map[j], n = p.n, nt = t.n;
  const double alpha = r.alpha[b], mu = p.mu[b];
  double pht = t.ft[j], tht = 0.0;
  for (long long i = 0; i < m; i++) {
    const long long e = i * n + b;
    const double gi = t.gt[i * nt + j], lo = p.lb[e], up = p.ub[e];
    if (kino::step_is_eq(i)) {
      tht += fabs(gi - lo);
      continue;
    }
    const double st = p.s[e] + alpha * r.ds[e];
    tht += fabs(gi - st);
    if (finite_lo(lo)) pht -= mu * log(st - lo);
    if (finite_up(up)) pht -= mu * log(up - st);
  }
  const double th0 = p.th0[b], theta = r.th[b], phi = r.phi[b], dphi = r.dphi[b];
  const double theta_max = 1e4 * fmax(1.0, th0), theta_min = 1e-4 * fmax(1.0, th0);
  bool ok = isfinite(pht) && isfinite(tht) && tht <= theta_max;
  for (int k = 0, nf = p.nfilt[b]; ok && k < nf; k++)
    if (tht >= p.fth[k * n + b] && pht >= p.fph[k * n + b]) ok = false;
  bool acc = false;
  int ftype = 0;
  if (ok) {
    const bool sw = (theta <= theta_min) && (dphi < 0) && (alpha * pow(-dphi, 2.3) > 1.0 * pow(theta, 1.1));
    if (sw) {
      if (pht <= phi + 1e-8 * alpha * dphi) { acc = true; ftype = 1; }
    } else if (tht <= (1.0 - 1e-5) * theta || pht <= phi - 1e-5 * theta) {
      acc = true;
    }
  }
  if (!acc) {
    const double a = alpha * 0.5;
    const int ls = r.ls[b] + 1;
    r.alpha[b] = a; r.ls[b] = ls;
    r.srch[b] = (a > 1e-12 * r.apr[b] && ls < 40) ? 1 : 0;
    return;
  }
  r.srch[b] = 0;
  const int tiny = alpha < o.jam_alpha ? p.tiny[b] + 1 : 0;
  p.tiny[b] = tiny;
  if (o.jam_iters > 0 && tiny >= o.jam_iters && p.rest[b] < o.max_restarts) return;  // watchdog: re-centre instead
  r.acc[b] = 1; r.ftype[b] = ftype;
  for (long long i = 0; i < nx; i++) p.x[i * n + b] = t.xt[i * nt + j];
  for (long long i = 0; i < m; i++) p.g[i * n + b] = t.gt[i * nt + j];
  p.f[b] = t.ft[j];
}

// accept (s, y, zL, zU with the kappa_sigma clamp, filter entry) or re-centre after a failed line search
__global__ void k_ks_accept(PS p, RS r, long long m, Opt o) {
  const long long b = (long long)blockIdx.x * NT + threadIdx.x;
  if (b >= p.n || p.status[b] != LANDING_ST_RUNNING) return;
  const long long n = p.n;
  if (!r.acc[b]) {
    p.tiny[b] = 0;
    if (p.rest[b] < o.max_restarts) {
      p.rest[b] += 1;
      const double mu = o.restart_mu > 0.0 ? o.restart_mu : o.mu_init;
      p.mu[b] = mu;
      init_slacks(p, b, m, o, mu);
      p.nfilt[b] = 0;
      p.th0[b] = -1.0;
      p.iters[b] += 1;
    } else {
      p.status[b] = LANDING_ST_LINESEARCH_FAIL;
    }
    return;
  }
  const double theta = r.th[b], phi = r.phi[b];
  if (!r.ftype[b]) {
    int nf = p.nfilt[b];
    if (nf == MAXF) {  // drop the oldest entry
      for (int k = 0; k < MAXF - 1; k++) {
        p.fth[k * n + b] = p.fth[(k + 1) * n + b];
        p.fph[k * n + b] = p.fph[(k + 1) * n + b];
      }
      nf--;
    }
    p.fth[nf * n + b] = (1.0 - 1e-5) * theta;
    p.fph[nf * n + b] = phi - 1e-5 * theta;
    p.nfilt[b] = nf + 1;
  }
  const double alpha = r.alpha[b], adu = r.adu[b], mu = p.mu[b], ks = 1e10;
  for (long long i = 0; i < m; i++) {
    const long long e = i * n + b;
    if (kino::step_is_eq(i)) {
      p.y[e] += alpha * r.dy[e];
      continue;
    }
    const double s = p.s[e] + alpha * r.ds[e], lo = p.lb[e], up = p.ub[e];
    p.s[e] = s;
    p.y[e] += alpha * r.dy[e];
    if (finite_lo(lo)) {
      const double d = s - lo;
      const double z = p.zL[e] + adu * r.dzL[e];
      p.zL[e] = fmax(fmin(z, ks * mu / d), mu / (ks * d));
    }
    if (finite_up(up)) {
      const double d = up - s;
      const double z = p.zU[e] + adu * r.dzU[e];
      p.zU[e] = fmax(fmin(z, ks * mu / d), mu / (ks * d));
    }
  }
  p.iters[b] += 1;
}

unsigned blocks(long long n) { return (unsigned)((n + NT - 1) / NT); }
unsigned rows_grid(long long rows) { return (unsigned)(rows < 1024 ? rows : 1024); }

}  // namespace

static long long kino_solve_doubles(int N, long long nnzJ, long long nnzH) {
  const Dims D{N, 12LL * N + 36LL * (N - 1), 48 + (long long)kino::ROWS_INT * (N - 2) + kino::ROWS_LAST, nnzJ, nnzH};
  return 2 * D.pd() + D.rd() + D.td();
}
static long long kino_solve_ints() { return 2 * PI_ROWS + RI_ROWS + 1; }
long long kino_solve_bytes(int N, long long nnzJ, long long nnzH) {
  return 8 * kino_solve_doubles(N, nnzJ, nnzH) + 4 * kino_solve_ints();
}

int kino_solve_run(const KinoSolveArgs& a, cudaStream_t st, long long* launches, long long stats[3], std::string* err) {
  const long long B = a.B;
  const Dims D{a.N, a.nx, a.m, a.nnzJ, a.nnzH};
  const long long nx = a.nx, m = a.m;
  // scratch: two persistent copies, the round, the trial points (doubles); their int rows; the map, the count
  double* Pd[2] = {a.scratch, a.scratch + D.pd() * B};
  double* Rd = Pd[1] + D.pd() * B;
  double* Td = Rd + D.rd() * B;
  int* Pi[2] = {reinterpret_cast<int*>(Td + D.td() * B), nullptr};
  Pi[1] = Pi[0] + PI_ROWS * B;
  int* Ri = Pi[1] + PI_ROWS * B;
  int* map = Ri + RI_ROWS * B;
  int* dcount = a.counter + 1;
  const double* ones = a.ones;
  const Opt o{a.opt.max_iter, a.opt.jam_iters, a.opt.max_restarts, a.opt.tol, a.opt.constr_viol_tol, a.opt.dual_inf_tol,
              a.opt.compl_inf_tol, a.opt.mu_init, a.opt.bound_push, a.opt.bound_frac, a.opt.bound_relax_factor,
              a.opt.jam_alpha, a.opt.restart_mu};
  const Out out{a.x_star, a.f_star, a.lam_g, a.viol, a.dual_inf, a.compl_inf, a.status, a.iters, a.restarts};
  long long L = 0, R = 0, S = 0, C = 0;
  auto check = [&](const char* what) -> int {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { *err = std::string(what) + ": " + cudaGetErrorString(e); return LANDING_ERR_CUDA; }
    return LANDING_OK;
  };
  auto read_count = [&](int* host) -> int {
    cudaError_t e = cudaMemcpyAsync(host, dcount, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { *err = std::string("kino solve read-back: ") + cudaGetErrorString(e); return LANDING_ERR_CUDA; }
    return LANDING_OK;
  };
  const CView ONE{ones, 0, 0};
  // ---- start: bounds (and the guess) of the drops, g and f at x0, slacks and multipliers
  long long Bc = B;
  int cur = 0;
  {
    const PS p = make_ps(Pd[0], Pi[0], B, D);
    KinoSetupArgs sa{};
    sa.N = a.N; sa.B = B; sa.ks = a.ks;
    sa.drops = make_cview(a.drops, 12, B, LANDING_AOS);
    sa.x_srb = make_cview(a.x_srb, 36LL * a.N - 24, B, LANDING_AOS);
    sa.lbg = View{p.lbo, B, 1}; sa.ubg = View{p.ubo, B, 1};
    sa.x0 = a.x0 ? View{nullptr, 0, 0} : View{p.x, B, 1};
    L += launch_kino_setup(sa, st);
    if (a.x0) { k_ks_load<<<dim3(blocks(B), rows_grid(nx)), NT, 0, st>>>(p, a.x0, nx); L++; }
    KinoArgs ka{};
    ka.N = a.N; ka.B = B; ka.x = CView{p.x, B, 1}; ka.g = View{p.g, B, 1}; ka.pr = a.pr; ka.dtv = a.dtv;
    ka.gpos = a.gpos; ka.bpos = a.bpos;
    L += launch_kino(ka, true, false, st);
    KinoSetupArgs ca{};
    ca.N = a.N; ca.B = B; ca.ks = a.ks; ca.x = CView{p.x, B, 1}; ca.f = View{p.f, B, 1};
    L += launch_kino_cost(ca, st);
    k_ks_init<<<blocks(B), NT, 0, st>>>(p, m, o);
    L++;
    if (int rc = check("kino solve start")) return rc;
  }
  for (;;) {
    R++;
    PS p = make_ps(Pd[cur], Pi[cur], Bc, D);
    RS r = make_rs(Rd, Ri, Bc, D);
    // ---- 1. grad_x of the Lagrangian (lam_f = 1, lam_g = y) and the final measures at x
    {
      KinoGradArgs ga{};
      ga.N = a.N; ga.B = Bc; ga.x = CView{p.x, Bc, 1}; ga.lam_f = ONE; ga.lam_g = CView{p.y, Bc, 1};
      ga.grad = View{r.gl, Bc, 1}; ga.pr = a.pr; ga.dtv = a.dtv;
      for (int i = 0; i < 12; i++) { ga.QN[i] = a.ks.QN[i]; ga.ref[i] = i < 6 ? a.ks.q_term_ref[i] : a.ks.qd_term_ref[i - 6]; }
      L += launch_kino_grad(ga, st);
      KinoKktArgs kk{};
      kk.B = Bc; kk.m = m; kk.nx = nx; kk.x = CView{p.x, Bc, 1}; kk.lam_f = ONE; kk.lam_g = CView{p.y, Bc, 1};
      kk.lbg = CView{p.lbo, Bc, 1}; kk.ubg = CView{p.ubo, Bc, 1}; kk.g = View{p.g, Bc, 1}; kk.grad = View{r.gl, Bc, 1};
      kk.viol = View{r.fv, Bc, 1}; kk.dual_inf = View{r.fd, Bc, 1}; kk.compl_inf = View{r.fc, Bc, 1};
      L += launch_kino_kkt(kk, st);
    }
    // ---- 2. measures, termination, barrier update
    k_ks_measure<<<blocks(Bc), NT, 0, st>>>(p, r, m, nx, o);
    k_ks_scan<<<1, SCAN_NT, 0, st>>>(p.status, LANDING_ST_RUNNING, Bc, map, dcount);
    L += 2;
    if (int rc = check("kino solve measure")) return rc;
    if (int rc = read_count(a.host_count)) return rc;
    const long long nrun = *a.host_count;
    if (nrun < Bc) {  // results of the finished scenarios out, the running ones to the front of the other copy
      C++;
      const PS q = make_ps(Pd[cur ^ 1], Pi[cur ^ 1], nrun, D);
      k_ks_output<<<dim3(blocks(Bc), rows_grid(nx + m)), NT, 0, st>>>(p, r, nx, m, out);
      L++;
      if (nrun > 0) {
        k_ks_gather<double><<<dim3(blocks(nrun), rows_grid(D.pd())), NT, 0, st>>>(Pd[cur], Bc, Pd[cur ^ 1], nrun, D.pd(), map);
        k_ks_gather<int><<<dim3(blocks(nrun), PI_ROWS), NT, 0, st>>>(Pi[cur], Bc, Pi[cur ^ 1], nrun, PI_ROWS, map);
        L += 2;
      }
      if (int rc = check("kino solve compaction")) return rc;
      cur ^= 1;
      Bc = nrun;
      p = q;
      r = make_rs(Rd, Ri, Bc, D);
    }
    if (Bc == 0) break;
    // ---- 3. Jacobian, cost gradient and Hessian (lam_f = 1, lam_g = y) of the running scenarios, and the Newton step
    {
      KinoArgs ka{};
      ka.N = a.N; ka.B = Bc; ka.x = CView{p.x, Bc, 1}; ka.jac = View{r.jac, Bc, 1}; ka.pr = a.pr; ka.dtv = a.dtv;
      ka.gpos = a.gpos; ka.bpos = a.bpos;
      L += launch_kino(ka, false, true, st);
      KinoSetupArgs ca{};
      ca.N = a.N; ca.B = Bc; ca.ks = a.ks; ca.x = CView{p.x, Bc, 1}; ca.grad_f = View{r.gf, Bc, 1};
      L += launch_kino_cost(ca, st);
      KinoHessArgs ha{};
      ha.N = a.N; ha.B = Bc; ha.x = CView{p.x, Bc, 1}; ha.lam_f = ONE; ha.lam_g = CView{p.y, Bc, 1};
      ha.hess = View{r.hess, Bc, 1}; ha.pr = a.pr; ha.dtv = a.dtv; ha.hpos = a.hpos; ha.cpos = a.cpos; ha.rows = a.hrows;
      for (int i = 0; i < 12; i++) ha.QN[i] = a.ks.QN[i];
      L += launch_kino_hess(ha, st);
    }
    {
      KinoStepArgs sa{};
      sa.B = Bc; sa.tb = a.tb;
      sa.g = CView{p.g, Bc, 1}; sa.jac = CView{r.jac, Bc, 1}; sa.hess = CView{r.hess, Bc, 1}; sa.grad_f = CView{r.gf, Bc, 1};
      sa.s = CView{p.s, Bc, 1}; sa.y = CView{p.y, Bc, 1}; sa.zL = CView{p.zL, Bc, 1}; sa.zU = CView{p.zU, Bc, 1};
      sa.lbg = CView{p.lb, Bc, 1}; sa.ubg = CView{p.ub, Bc, 1}; sa.mu = CView{p.mu, Bc, 1}; sa.dw_last = CView{p.dwl, Bc, 1};
      sa.dx = View{r.dx, Bc, 1}; sa.ds = View{r.ds, Bc, 1}; sa.dy = View{r.dy, Bc, 1}; sa.dzL = View{r.dzL, Bc, 1};
      sa.dzU = View{r.dzU, Bc, 1}; sa.delta_w = View{r.dw, Bc, 1};
      sa.alpha_pr = View{nullptr, 0, 0}; sa.alpha_du = View{nullptr, 0, 0};
      sa.n_factor = r.nf; sa.status = r.sst; sa.tau = 0.0;
      sa.scratch = a.step_scr; sa.slot = a.step_slot; sa.counter = a.counter;
      if (cudaMemsetAsync(a.counter, 0, sizeof(int), st) != cudaSuccess) return check("kino solve step counter");
      L += launch_kino_step(sa, (int)(Bc < a.step_grid ? Bc : a.step_grid), st);
    }
    // ---- 4. fraction to the boundary, merit
    k_ks_ftb<<<blocks(Bc), NT, 0, st>>>(p, r, m, a.N);
    L++;
    // ---- 5. line search over the scenarios still searching
    for (;;) {
      k_ks_scan<<<1, SCAN_NT, 0, st>>>(r.srch, 1, Bc, map, dcount);
      L++;
      if (int rc = check("kino solve line search")) return rc;
      if (int rc = read_count(a.host_count)) return rc;
      const long long ns = *a.host_count;
      if (ns == 0) break;
      S++;
      const TS t = make_ts(Td, ns, D);
      k_ks_trial<<<dim3(blocks(ns), rows_grid(nx)), NT, 0, st>>>(p, r, t, nx, map);
      KinoArgs ka{};
      ka.N = a.N; ka.B = ns; ka.x = CView{t.xt, ns, 1}; ka.g = View{t.gt, ns, 1}; ka.pr = a.pr; ka.dtv = a.dtv;
      ka.gpos = a.gpos; ka.bpos = a.bpos;
      L += 1 + launch_kino(ka, true, false, st);
      KinoSetupArgs ca{};
      ca.N = a.N; ca.B = ns; ca.ks = a.ks; ca.x = CView{t.xt, ns, 1}; ca.f = View{t.ft, ns, 1};
      L += launch_kino_cost(ca, st);
      k_ks_filter<<<blocks(ns), NT, 0, st>>>(p, r, t, nx, m, o, map);
      L++;
    }
    // ---- 6. accept or re-centre
    k_ks_accept<<<blocks(Bc), NT, 0, st>>>(p, r, m, o);
    L++;
    if (int rc = check("kino solve accept")) return rc;
  }
  *launches += L;
  stats[0] = R; stats[1] = S; stats[2] = C;
  return LANDING_OK;
}

}  // namespace srb
