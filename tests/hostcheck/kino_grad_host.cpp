// tests/hostcheck/kino_grad_host.cpp -- TEST HARNESS (CPU): compiles the owner contraction of the kino-dynamic
// Lagrangian gradient (landing_controller_b200/csrc/kino_grad.cuh) for the host, so that it can be checked against the
// oracle's exact Jacobian without a GPU.  Not part of the product library and never used as a fallback.
#include <utility>

#include "../../landing_controller_b200/csrc/kino_grad.cuh"

using namespace srb::kino;

static Params params(const double* prm) {  // mu, mass, Ib[3], Ib_inv[3]
  return Params{prm[0], prm[1], {prm[2], prm[3], prm[4]}, {prm[5], prm[6], prm[7]}};
}

// The kernels' contraction: acc[j] += lam_g[row] * tangent j (fma, as on the device), and the boundary identities.
struct LamCtr {
  const double* lam;
  double acc[3];
  void operator()(long long row, const DualN<3>& v) {
    for (int j = 0; j < 3; j++) acc[j] = __builtin_fma(lam[row], v.d[j], acc[j]);
  }
  void ident(long long row, int j) { acc[j] += lam[row]; }
};

// Instrumented contraction: every (row, column) pair the owner touches, cnt[row * nx + col] += 1, and nz[...] += 1 where
// the tangent it contracts is non-zero.
struct CoverCtr {
  long long nx, col0;
  int *cnt, *nz;
  void operator()(long long row, const DualN<3>& v) {
    for (int j = 0; j < 3; j++) {
      cnt[row * nx + col0 + j] += 1;
      nz[row * nx + col0 + j] += v.d[j] != 0.0;
    }
  }
  void ident(long long row, int j) {
    cnt[row * nx + col0 + j] += 1;
    nz[row * nx + col0 + j] += 1;
  }
};

struct Problem {
  int N;
  const double *x, *dt;
  Params pr;
};

// every owner of the batch's one scenario: triples T of knots 0..N-1 (X) or 0..N-2 (jpos, U)
template <int T, class F>
static void owners(const Problem& p, F&& f) {
  for (int k = 0; k < (T < 4 ? p.N : p.N - 1); k++) f(std::integral_constant<int, T>{}, k, knot_col(p.N, k, 3 * T));
}
template <class F, int... T>
static void all_owners(const Problem& p, F&& f, std::integer_sequence<int, T...>) {
  (owners<T>(p, f), ...);
}

// grad[nx] = lam_f grad f + J' lam_g, owner by owner as the kernels compute it
extern "C" int kino_grad_host(int N, const double* x, const double* dt, const double* prm, const double* lam_g,
                              double lam_f, const double* QN, const double* ref, double* grad) {
  const Problem p{N, x, dt, params(prm)};
  auto ld = [&](long long col) { return x[col]; };
  all_owners(p, [&](auto t, int k, long long col0) {
    constexpr int T = decltype(t)::value;
    LamCtr c{lam_g, {0.0, 0.0, 0.0}};
    grad_rows<T>(N, k, ld, dt, p.pr, c);
    grad_cost<T>(N, k, ld, lam_f, QN, ref, c.acc);
    for (int j = 0; j < 3; j++) grad[col0 + j] = c.acc[j];
  }, std::make_integer_sequence<int, GRAD_TRIPLES>{});
  return 0;
}

// cnt, nz [m x nx] (zeroed by the caller)
extern "C" int kino_grad_cover(int N, const double* x, const double* dt, const double* prm, int* cnt, int* nz) {
  const Problem p{N, x, dt, params(prm)};
  const long long nx = 12LL * N + 36LL * (N - 1);
  auto ld = [&](long long col) { return x[col]; };
  all_owners(p, [&](auto t, int k, long long col0) {
    constexpr int T = decltype(t)::value;
    CoverCtr c{nx, col0, cnt, nz};
    grad_rows<T>(N, k, ld, dt, p.pr, c);
  }, std::make_integer_sequence<int, GRAD_TRIPLES>{});
  return 0;
}
