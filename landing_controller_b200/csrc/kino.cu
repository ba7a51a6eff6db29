// kino.cu -- batched evaluation of the kino-dynamic ("full-body") landing NLP of the reference's KNITRO variant
// (SURVEY 8 f-2; generate_solver/generate_landingCtrller_KNITRO.m:34-193): constraint values g and the sparse Jacobian
// dg/dx in CCS order for a whole batch of trajectories.  One thread = one (scenario, knot); with the SoA layout every
// load and store of a warp is one coalesced 256-byte transaction.  The Jacobian columns are exact forward-mode
// derivatives of the same knot function (kino_knot.cuh, DualN): one pass per triple of knot-local inputs, each pass its
// own thread; a pass types only its own input block as duals and evaluates only the row groups it can reach.  Bounds,
// initial guess and terminal cost of the same NLP: k_kino_setup, k_kino_cost.
//
// x = [X(:) (12 N); jpos(:) (12 (N-1)); U(:) (24 (N-1))], g rows: 48 boundary rows, then 141 per knot (117 for the
// last) -- the row map is in oracle/kino_ref.py, which is pinned to the solution of this NLP that the reference stores.
#include <algorithm>
#include <map>
#include <random>
#include <vector>

#include "kernels.cuh"
#include "kino_knot.cuh"

namespace srb {
namespace {

using kino::Dual1;
using kino::NIN;
using kino::ROWS_INT;
using kino::ROWS_LAST;

struct GSink {
  View g;
  long long b, base;
  __device__ __forceinline__ void operator()(int rho, double v) { g.at(base + rho, b) = v; }
};
// Sink of a Jacobian pass: a row whose value is a plain double does not depend on the seeded block (no entry); a dual
// row scatters its K tangents to the CCS positions of (row, seeded columns) from the host-made table (-1 = no entry).
template <int K> struct JSinkN {
  View jac;
  long long b;
  const int* gp;  // table row of the first seeded input: gp[j * ROWS_INT + rho]
  __device__ __forceinline__ void operator()(int, double) const {}
  __device__ __forceinline__ void operator()(int rho, const kino::DualN<K>& v) const {
#pragma unroll
    for (int j = 0; j < K; j++) {
      const int p = __ldg(gp + j * ROWS_INT + rho);
      if (p >= 0) jac.at(p, b) = v.d[j];
    }
  }
};

// One (scenario, knot) is evaluated by four threads of four different CTAs (blockIdx.z = part = leg): each runs the whole
// knot function behind a compile-time filtering sink and emits only the rows its part owns (kino::row_owner), so the
// compiler removes the other legs' kinematics from its instance -- the same device the SRB evaluation kernels use
// (eval.cu: PartSink).  Four times the threads in flight, a third of the work each.
template <bool LAST, int PART> struct GPartSink {
  View g;
  long long b, base;
  __device__ __forceinline__ void operator()(int rho, double v) {
    if (kino::row_owner<LAST>(rho) == PART) g.at(base + rho, b) = v;
  }
};
template <bool LAST, int PART>
__device__ __forceinline__ void kino_g_part(const KinoArgs& a, long long b, int k) {
  double in[NIN];  // (loaded here, per instance: the loads of inputs a part never uses are dead code)
#pragma unroll
  for (int v = 0; v < NIN; v++) in[v] = (LAST && v >= 60) ? 0.0 : a.x.get(kino_col(a.N, k, v), b);
  GPartSink<LAST, PART> s{a.g, b, 48 + (long long)ROWS_INT * k};
  kino::knot_rows_t<LAST, double>(in, __ldg(a.dtv + k), a.pr, s,
                                  (kino::G_LEG0 << PART) | (PART == 0 ? (kino::G_DYN | kino::G_FRIC | kino::G_Z) : 0u) | kino::G_JPOS);
}

#ifndef KINO_G_CTAS
#define KINO_G_CTAS 4  // (128 registers: 0.159 ms instead of 0.165 ms at 16k scenarios, N = 21; 5 / 6 CTAs are slower)
#endif
__global__ void __launch_bounds__(128, KINO_G_CTAS) k_kino_g(KinoArgs a) {
  const long long b = (long long)blockIdx.x * 128 + threadIdx.x;
  if (b >= a.B) return;
  const int N = a.N, k = blockIdx.y, part = blockIdx.z;
  const bool last = k == N - 2;
  switch (part) {  // (block-uniform)
    case 0: if (last) kino_g_part<true, 0>(a, b, k); else kino_g_part<false, 0>(a, b, k); break;
    case 1: if (last) kino_g_part<true, 1>(a, b, k); else kino_g_part<false, 1>(a, b, k); break;
    case 2: if (last) kino_g_part<true, 2>(a, b, k); else kino_g_part<false, 2>(a, b, k); break;
    default: if (last) kino_g_part<true, 3>(a, b, k); else kino_g_part<false, 3>(a, b, k); break;
  }
  if (k == 0 && part == 0) {  // boundary rows: q_0, qd_0, c_0 | q_{N-1} twice | qd_{N-1} twice   (:93-101)
    for (int i = 0; i < 12; i++) a.g.at(i, b) = a.x.get(i, b);
    for (int i = 0; i < 12; i++) a.g.at(12 + i, b) = a.x.get(12LL * N + 12LL * (N - 1) + i, b);
    for (int i = 0; i < 6; i++) {
      const double q = a.x.get(12LL * (N - 1) + i, b), qd = a.x.get(12LL * (N - 1) + 6 + i, b);
      a.g.at(24 + i, b) = q; a.g.at(30 + i, b) = q;
      a.g.at(36 + i, b) = qd; a.g.at(42 + i, b) = qd;
    }
  }
}

// Jacobian: the passes of kino_knot.cuh (kino::PassOf, kino::jac_pass), one thread per (scenario, knot, pass).
template <bool LAST, int G>
__device__ __forceinline__ void kino_jac_pass(const KinoArgs& a, long long b, int k) {
  double x[NIN];  // (loads of inputs the pass never uses are dead code)
#pragma unroll
  for (int v = 0; v < NIN; v++) x[v] = (LAST && v >= 60) ? 0.0 : a.x.get(kino_col(a.N, k, v), b);
  const double h = __ldg(a.dtv + k);
  JSinkN<3> s{a.jac, b, a.gpos + ((long long)k * NIN + kino::PassOf<G>::v0) * ROWS_INT};
  kino::jac_pass<LAST, G>(x, h, a.pr, s);
}
template <bool LAST, int G, int G1>
__device__ __forceinline__ void kino_jac_dispatch(const KinoArgs& a, long long b, int k, int g) {
  if constexpr (G < G1) {
    if (g == G) {
      if constexpr (kino::pass_in_knot(LAST, G)) kino_jac_pass<LAST, G>(a, b, k);
    } else {
      kino_jac_dispatch<LAST, G + 1, G1>(a, b, k, g);
    }
  }
}

// Passes G0..G1-1; blockIdx.x = pass + (G1 - G0) * scenario block: the passes of one (scenario block, knot) read the same
// x and are scheduled together, so all but the first find it in L2.  One kernel per class of passes (launch_kino), so
// that the light passes are not held to the register count -- hence occupancy -- of the rpy passes.
// Six CTAs per SM (80 registers; a few hundred bytes of spills in the rpy-leg passes): the passes are bound by the latency
// of their dependent FP64 chains, not by arithmetic or bandwidth.  Measured at 16k scenarios, N = 21: no cap 1.07 ms, 5 CTAs
// 0.99, 6 CTAs 0.95, 8 CTAs 1.12.  Both neighbours of this organisation were measured slower: the five passes of a leg
// in ONE thread on one copy of x and one evaluation of the sincos (1.22 ms) and a finer split of the r / c / f triples
// into dynamics and leg passes (40 passes: 1.21 ms).
#ifndef KINO_JAC_CTAS
#define KINO_JAC_CTAS 6
#endif
template <int G0, int G1>
__global__ void __launch_bounds__(128, KINO_JAC_CTAS) k_kino_jac(KinoArgs a) {
  constexpr int NPASS = G1 - G0;
  const int g = G0 + (int)(blockIdx.x % NPASS);
  const long long b = (long long)(blockIdx.x / NPASS) * 128 + threadIdx.x;
  if (b >= a.B) return;
  const int N = a.N, k = blockIdx.y;  // (block-uniform dispatch)
  if (k == N - 2) kino_jac_dispatch<true, G0, G1>(a, b, k, g);
  else kino_jac_dispatch<false, G0, G1>(a, b, k, g);
  if (G0 == 0 && k == 0 && g == 0)
    for (int i = 0; i < 48; i++) a.jac.at(__ldg(a.bpos + i), b) = 1.0;
}

// ---------------------------------------------------------------- bounds, initial guess, terminal cost
// (generate_landingCtrller_KNITRO.m:198-262,300-327; include/landing_b200.h: landing_kino_setup_batch)
__device__ __forceinline__ void rot_xyz(const double* rpy, double* R) {  // rpyToRotMat_xyz.m:2, body -> world, row-major
  double sr, cr, sp, cp, sy, cy;
  sincos(rpy[0], &sr, &cr);
  sincos(rpy[1], &sp, &cp);
  sincos(rpy[2], &sy, &cy);
  R[0] = cp * cy; R[1] = -(cp * sy); R[2] = sp;
  R[3] = cr * sy + sr * sp * cy; R[4] = cr * cy - sr * sp * sy; R[5] = -(sr * cp);
  R[6] = sr * sy - cr * sp * cy; R[7] = sr * cy + cr * sp * sy; R[8] = cr * cp;
}
__device__ __forceinline__ double foot_sx(int l) { return l < 2 ? 1.0 : -1.0; }   // sideSign of :200 (x, y; z = 1)
__device__ __forceinline__ double foot_sy(int l) { return (l & 1) ? 1.0 : -1.0; }
__device__ __forceinline__ double kin_box_limit(double v, double bmax) {           // utilities_landing/kin_box_limits.m
  return fabs(v) < 2.0 ? fabs(v * bmax / 2.0) : bmax;
}

__global__ void __launch_bounds__(128) k_kino_setup(KinoSetupArgs a) {
  const long long b = (long long)blockIdx.x * 128 + threadIdx.x;
  if (b >= a.B) return;
  const int N = a.N, k = blockIdx.y;
  const landing_kino_setup& ks = a.ks;
  const double INF = HUGE_VAL;
  double q0[6], qd0[6], R0[9];
#pragma unroll
  for (int i = 0; i < 6; i++) { q0[i] = a.drops.get(i, b); qd0[i] = a.drops.get(6 + i, b); }
  rot_xyz(q0 + 3, R0);
  auto set = [&](long long row, double l, double u) {
    if (a.lbg.p) a.lbg.at(row, b) = l;
    if (a.ubg.p) a.ubg.at(row, b) = u;
  };
  // state of knot k of the initial guess: the SRB solution, else the reference trajectory (:272-275)
  double Xk[12];
  if (a.x0.p) {
    const double t = (double)k / (double)(N - 1);
#pragma unroll
    for (int i = 0; i < 12; i++) {
      const double from = i < 6 ? q0[i] : qd0[i - 6], to = i < 6 ? ks.q_term_ref[i] : ks.qd_term_ref[i - 6];
      Xk[i] = a.x_srb.p ? a.x_srb.get(12LL * k + i, b) : from + (to - from) * t;
      a.x0.at(12LL * k + i, b) = Xk[i];
    }
  }
  if (k == N - 1) {  // boundary rows (:93-101)
    if (a.lbg.p || a.ubg.p) {
#pragma unroll
      for (int i = 0; i < 6; i++) {
        set(i, q0[i], q0[i]);
        set(6 + i, qd0[i], qd0[i]);
        set(24 + i, ks.q_term_min[i], INF);
        set(30 + i, -INF, ks.q_term_max[i]);
        set(36 + i, ks.qd_term_min[i], INF);
        set(42 + i, -INF, ks.qd_term_max[i]);
      }
#pragma unroll
      for (int l = 0; l < 4; l++) {  // c_init (:232-236)
        const double p[3] = {foot_sx(l) * 0.2, foot_sy(l) * 0.15, -0.3};
#pragma unroll
        for (int i = 0; i < 3; i++) {
          const double c = q0[i] + R0[3 * i] * p[0] + R0[3 * i + 1] * p[1] + R0[3 * i + 2] * p[2];
          set(12 + 3 * l + i, c, c);
        }
      }
    }
    return;
  }
  if (a.x0.p) {
    const long long jo = 12LL * N + 12LL * k, uo = 12LL * N + 12LL * (N - 1) + 24LL * k;
#pragma unroll
    for (int i = 0; i < 12; i++) a.x0.at(jo + i, b) = ks.jpos_guess[i % 3];  // (:325)
    if (a.x_srb.p) {
      for (int i = 0; i < 24; i++) a.x0.at(uo + i, b) = a.x_srb.get(12LL * N + 24LL * k + i, b);
    } else {  // Uref (:276-286): reference feet under the reference body, no force
      double Rk[9];
      rot_xyz(Xk + 3, Rk);
#pragma unroll
      for (int l = 0; l < 4; l++) {
        const double p[3] = {foot_sx(l) * 0.2, foot_sy(l) * 0.2, -0.3};
#pragma unroll
        for (int i = 0; i < 3; i++) {
          a.x0.at(uo + 3 * l + i, b) = Xk[i] + Rk[3 * i] * p[0] + Rk[3 * i + 1] * p[1] + Rk[3 * i + 2] * p[2];
          a.x0.at(uo + 12 + 3 * l + i, b) = 0.0;
        }
      }
    }
  }
  if (!a.lbg.p && !a.ubg.p) return;
  // kinematic box from the body-frame velocity of the drop (:246-248)
  const double vb0 = R0[0] * qd0[3] + R0[3] * qd0[4] + R0[6] * qd0[5], vb1 = R0[1] * qd0[3] + R0[4] * qd0[4] + R0[7] * qd0[5];
  const double kx = 0.125 + kin_box_limit(vb0, 0.15), ky = 0.125 + kin_box_limit(vb1, 0.25);
  const bool last = k == N - 2;
  const long long base = 48 + (long long)ROWS_INT * k;
  for (int i = 0; i < 12; i++) set(base + i, 0.0, 0.0);        // dynamics (:128-131)
  for (int l = 0; l < 4; l++) set(base + 12 + l, 0.0, INF);    // f_z >= 0 (:134)
  const int per_leg = last ? 9 : 15;
  for (int l = 0; l < 4; l++) {
    long long r = base + 16 + per_leg * l;
    set(r++, 0.0, INF);          // c_z >= 0 (:141)
    set(r++, -INF, 0.001);       // f_z c_z <= 0.001 (:142)
    if (!last) {
      for (int i = 0; i < 3; i++) set(r++, -INF, 0.001);   // no-slip (:145-146)
      for (int i = 0; i < 3; i++) set(r++, -0.001, INF);
    }
    set(r++, -kx, kx);                                      // kinematic box (:161-167)
    if ((l & 1) == 0) set(r++, -ky, 0.05); else set(r++, -0.05, ky);
    set(r++, -0.4, -0.075);
    set(r++, -INF, ks.l_leg_max * ks.l_leg_max);            // leg length (:168)
    for (int i = 0; i < 3; i++) set(r++, -ks.tau_max[i], ks.tau_max[i]);  // torques (:173-175)
  }
  long long r = base + 16 + 4 * per_leg;
  for (int i = 0; i < 16; i++) set(r++, -INF, 0.0);         // friction pyramid (:179-182)
  set(r++, ks.z_min, INF);                                  // z_k >= q_min(3) (:185)
  for (int i = 0; i < 12; i++) set(r++, -0.01, INF);        // c - FK (:190-191)
  for (int i = 0; i < 12; i++) set(r++, -INF, 0.01);
  for (int i = 0; i < 12; i++) set(r++, ks.jpos_min[i], INF);  // joint limits (:192-193)
  for (int i = 0; i < 12; i++) set(r++, -INF, ks.jpos_max[i]);
}

// f = (X_N - Xref_N)' QN (X_N - Xref_N) (:86-88); grad_f is pre-zeroed by the launcher
__global__ void __launch_bounds__(128) k_kino_cost(KinoSetupArgs a) {
  const long long b = (long long)blockIdx.x * 128 + threadIdx.x;
  if (b >= a.B) return;
  const long long xo = 12LL * (a.N - 1);
  double fv = 0.0;
#pragma unroll
  for (int i = 0; i < 12; i++) {
    const double d = a.x.get(xo + i, b) - (i < 6 ? a.ks.q_term_ref[i] : a.ks.qd_term_ref[i - 6]);
    fv += a.ks.QN[i] * d * d;
    if (a.grad_f.p) a.grad_f.at(xo + i, b) = 2.0 * a.ks.QN[i] * d;
  }
  if (a.f.p) a.f.at(0, b) = fv;
}

}  // namespace

// ---------------------------------------------------------------- host: pattern and CCS tables
KinoPlan make_kino_plan(int N) {
  KinoPlan pl;
  pl.N = N;
  pl.nx = 12LL * N + 36LL * (N - 1);
  pl.m = 48 + (long long)ROWS_INT * (N - 2) + ROWS_LAST;
  const int K = N - 1;
  // knot-local pattern by probing the knot function with tangents at random points (both knot classes)
  std::mt19937_64 rng(12345);
  std::uniform_real_distribution<double> U(-1.0, 1.0);
  kino::Params pr{0.75, 8.252, {0.0576, 0.234, 0.28}, {17.4, 4.27, 3.58}};
  std::vector<char> pat[2];
  for (int cls = 0; cls < 2; cls++) {
    const bool last = cls == 1;
    pat[cls].assign((size_t)NIN * ROWS_INT, 0);
    for (int rep = 0; rep < 3; rep++) {
      double xv[NIN];
      for (int i = 0; i < NIN; i++) xv[i] = U(rng);
      for (int v = 0; v < NIN; v++) {
        if (last && v >= 60) continue;
        Dual1 in[NIN];
        for (int i = 0; i < NIN; i++) in[i] = Dual1(xv[i], i == v ? 1.0 : 0.0);
        auto sink = [&](int rho, Dual1 d) { if (d.d[0] != 0.0) pat[cls][(size_t)v * ROWS_INT + rho] = 1; };
        kino::knot_rows<Dual1>(in, 0.03, pr, last, sink);
      }
    }
  }
  // global entries (col, row) -> CCS order
  struct E { long long col, row; int k, v, rho; };
  std::vector<E> ent;
  auto bnd = [&](int row, long long col) { ent.push_back({col, row, -1, row, 0}); };
  for (int i = 0; i < 12; i++) bnd(i, i);
  for (int i = 0; i < 12; i++) bnd(12 + i, 12LL * N + 12LL * (N - 1) + i);
  for (int i = 0; i < 6; i++) {
    bnd(24 + i, 12LL * (N - 1) + i); bnd(30 + i, 12LL * (N - 1) + i);
    bnd(36 + i, 12LL * (N - 1) + 6 + i); bnd(42 + i, 12LL * (N - 1) + 6 + i);
  }
  for (int k = 0; k < K; k++) {
    const int cls = k == K - 1;
    for (int v = 0; v < NIN; v++)
      for (int rho = 0; rho < ROWS_INT; rho++)
        if (pat[cls][(size_t)v * ROWS_INT + rho]) ent.push_back({kino_col(N, k, v), 48 + (long long)ROWS_INT * k + rho, k, v, rho});
  }
  std::sort(ent.begin(), ent.end(), [](const E& a, const E& b) { return a.col != b.col ? a.col < b.col : a.row < b.row; });
  pl.nnz = (long long)ent.size();
  pl.sparsity.assign(2 + pl.nx + 1 + pl.nnz, 0);
  pl.sparsity[0] = pl.m; pl.sparsity[1] = pl.nx;
  pl.gpos.assign((size_t)K * NIN * ROWS_INT, -1);
  pl.bpos.assign(48, 0);
  for (long long p = 0; p < pl.nnz; p++) {
    const E& e = ent[p];
    pl.sparsity[2 + e.col + 1] += 1;
    pl.sparsity[2 + pl.nx + 1 + p] = e.row;
    if (e.k < 0) pl.bpos[e.v] = (int)p;
    else pl.gpos[((size_t)e.k * NIN + e.v) * ROWS_INT + e.rho] = (int)p;
  }
  for (long long c = 0; c < pl.nx; c++) pl.sparsity[2 + c + 1] += pl.sparsity[2 + c];
  return pl;
}

int launch_kino(const KinoArgs& a, bool want_g, bool want_jac, cudaStream_t st) {
  int n = 0;
  const unsigned gx = (unsigned)((a.B + 127) / 128);
  if (want_g) { k_kino_g<<<dim3(gx, a.N - 1, 4), 128, 0, st>>>(a); n++; }
  if (want_jac) {
    k_kino_jac<0, 1><<<dim3(gx * 1, a.N - 1, 1), 128, 0, st>>>(a);     // r
    k_kino_jac<1, 2><<<dim3(gx * 1, a.N - 1, 1), 128, 0, st>>>(a);     // rpy: dynamics rows
    k_kino_jac<2, 4><<<dim3(gx * 2, a.N - 1, 1), 128, 0, st>>>(a);     // omega, v
    k_kino_jac<4, 8><<<dim3(gx * 4, a.N - 1, 1), 128, 0, st>>>(a);     // joint angles by leg
    k_kino_jac<8, 12><<<dim3(gx * 4, a.N - 1, 1), 128, 0, st>>>(a);    // foot positions by leg
    k_kino_jac<12, 16><<<dim3(gx * 4, a.N - 1, 1), 128, 0, st>>>(a);   // forces by leg
    k_kino_jac<16, 24><<<dim3(gx * 8, a.N - 1, 1), 128, 0, st>>>(a);   // next state, next foot positions
    k_kino_jac<24, 28><<<dim3(gx * 4, a.N - 1, 1), 128, 0, st>>>(a);   // rpy: rows of one leg
    n += 8;
  }
  return n;
}

int launch_kino_setup(const KinoSetupArgs& a, cudaStream_t st) {
  k_kino_setup<<<dim3((unsigned)((a.B + 127) / 128), a.N, 1), 128, 0, st>>>(a);
  return 1;
}

int launch_kino_cost(const KinoSetupArgs& a, cudaStream_t st) {
  if (a.grad_f.p) cudaMemsetAsync(a.grad_f.p, 0, sizeof(double) * (12LL * a.N + 36LL * (a.N - 1)) * a.B, st);
  k_kino_cost<<<(unsigned)((a.B + 127) / 128), 128, 0, st>>>(a);
  return 1;
}

}  // namespace srb
