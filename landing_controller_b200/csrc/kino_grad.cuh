// kino_grad.cuh -- the Lagrangian gradient of the kino-dynamic NLP by column owner, host and device:
// grad_x = lam_f grad f + J' lam_g (CasADi nlp_grad: grad_gamma_x) without forming J.  The Jacobian passes of
// kino_knot.cuh (kino::PassOf, kino::jac_pass) run with a sink that contracts each dual row with lam_g in registers.
//
// Owners.  Column triple T of knot k (the knot-local inputs 3T..3T+2: T = 0 r, 1 rpy, 2 omega, 3 v of X_k, k = 0..N-1;
// 4 + l joint angles, 8 + l foot position, 12 + l force of leg l of jpos_k / U_k, k = 0..N-2) has one owner, which adds
// every contribution to its three columns in a fixed order:
//   1. knot k's own passes: G = T, and for rpy also G = 24..27 (its rows of each leg);
//   2. knot k-1's passes whose seeded triple is this one: X_k is X+ of knot k-1 (G = 16 + T), c_k is c+ of knot k-1
//      (G = 12 + T);
//   3. the boundary identities: q_0, qd_0 (rows 0..11), c_0 (rows 12..23), X_{N-1} twice (rows 24..47);
//   4. the terminal cost on X_{N-1} (grad_cost).
// X_{N-1} has no knot of its own: its owners run only knot N-2's X+ passes.  Each gradient entry therefore has one writer,
// no atomics and no scratch, and the sum is in the same order whatever the layout or memory space.
#pragma once
#include "kino_knot.cuh"

namespace srb {
namespace kino {

constexpr int GRAD_TRIPLES = 16;

// Sink of a Jacobian pass inside an owner: a plain double row does not depend on the seeded triple (nothing to add, and
// lam_g is not read); a dual row goes to the contraction c(global row, tangents).
template <class Ctr> struct GradSink {
  Ctr& c;
  long long base;
  KHD void operator()(int, double) const {}
  KHD void operator()(int rho, const DualN<3>& v) const { c(base + rho, v); }
};

// Knot-local inputs of knot kk through the loader ld(column).
template <bool LAST, class Ld>
KHD void load_knot(int N, int kk, const Ld& ld, double* x) {
#pragma unroll
  for (int v = 0; v < NIN; v++) x[v] = (LAST && v >= 60) ? 0.0 : ld(knot_col(N, kk, v));
}

template <bool LAST, int G, class Ctr>
KHD void grad_pass(const double* x, double h, const Params& pr, long long base, Ctr& c) {
  if constexpr (pass_in_knot(LAST, G)) {
    GradSink<Ctr> s{c, base};
    jac_pass<LAST, G>(x, h, pr, s);
  }
}

// 1: the passes of knot k that seed triple T
template <bool LAST, int T, class Ld, class Ctr>
KHD void grad_own(int N, int k, const Ld& ld, const double* dt, const Params& pr, Ctr& c) {
  double x[NIN];  // (loads of inputs the passes never use are dead code)
  load_knot<LAST>(N, k, ld, x);
  const double h = dt[k];
  const long long base = 48 + (long long)ROWS_INT * k;
  grad_pass<LAST, T>(x, h, pr, base, c);
  if constexpr (T == 1) {
    grad_pass<LAST, 24>(x, h, pr, base, c);
    grad_pass<LAST, 25>(x, h, pr, base, c);
    grad_pass<LAST, 26>(x, h, pr, base, c);
    grad_pass<LAST, 27>(x, h, pr, base, c);
  }
}

// 2: the pass of knot k - 1 that seeds triple T as X+ or c+
template <bool LAST, int T, class Ld, class Ctr>
KHD void grad_prev(int N, int k, const Ld& ld, const double* dt, const Params& pr, Ctr& c) {
  constexpr int G = T < 4 ? 16 + T : 12 + T;
  double x[NIN];
  load_knot<LAST>(N, k - 1, ld, x);
  grad_pass<LAST, G>(x, dt[k - 1], pr, 48 + (long long)ROWS_INT * (k - 1), c);
}

// J' lam_g on the columns of triple T of knot k: c(row, DualN<3>) for knot rows, c.ident(row, j) for the identity entry
// of a boundary row in column j of the triple.
template <int T, class Ld, class Ctr>
KHD void grad_rows(int N, int k, const Ld& ld, const double* dt, const Params& pr, Ctr& c) {
  if (k <= N - 2) {
    if (k == N - 2) grad_own<true, T>(N, k, ld, dt, pr, c);
    else grad_own<false, T>(N, k, ld, dt, pr, c);
  }
  if constexpr (T < 4 || (T >= 8 && T < 12)) {
    if (k >= 1) {
      if (k - 1 == N - 2) grad_prev<true, T>(N, k, ld, dt, pr, c);  // (only X_{N-1}: the last knot has no c+)
      else grad_prev<false, T>(N, k, ld, dt, pr, c);
    }
  }
  if constexpr (T < 4) {
    if (k == 0) {
#pragma unroll
      for (int j = 0; j < 3; j++) c.ident(3 * T + j, j);       // q_0, qd_0
    }
    if (k == N - 1) {                                          // q_{N-1} twice, qd_{N-1} twice
      constexpr int r0 = T < 2 ? 24 + 3 * T : 36 + 3 * (T - 2);
#pragma unroll
      for (int j = 0; j < 3; j++) c.ident(r0 + j, j);
#pragma unroll
      for (int j = 0; j < 3; j++) c.ident(r0 + 6 + j, j);
    }
  }
  if constexpr (T >= 8 && T < 12) {
    if (k == 0) {
#pragma unroll
      for (int j = 0; j < 3; j++) c.ident(12 + 3 * (T - 8) + j, j);  // c_0
    }
  }
}

// lam_f grad f on the columns of triple T of knot k: f = (X_{N-1} - ref)' QN (X_{N-1} - ref), the formula of
// k_kino_cost; acc[j] += lam_f (2 QN_i (x_i - ref_i)).
template <int T, class Ld>
KHD void grad_cost(int N, int k, const Ld& ld, double lam_f, const double* QN, const double* ref, double* acc) {
  if constexpr (T < 4) {
    if (k == N - 1) {
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const int i = 3 * T + j;
        acc[j] += lam_f * (2.0 * QN[i] * (ld(12LL * (N - 1) + i) - ref[i]));
      }
    }
  }
}

}  // namespace kino
}  // namespace srb
