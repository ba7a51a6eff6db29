// tests/hostcheck/kino_hess_host.cpp -- TEST HARNESS (CPU): compiles the product's kino-dynamic knot template
// (landing_controller_b200/csrc/kino_knot.cuh) for the host with the second-order scalar type, so that the Hessian pass
// table of the kernels (kino::hess_pair, kino::HessPassOf masks, kino::hess_pass seeding, the last-knot skip) can be
// checked against the oracle without a GPU.  Not part of the product library and never used as a fallback.
#include <utility>

#include "../../landing_controller_b200/csrc/kino_knot.cuh"

using namespace srb::kino;

// The pass table: pass -> triples (a, b) and whether it runs in the last knot.
extern "C" int kino_hess_host_table(int* a, int* b, int* in_last) {
  for (int P = 0; P < HESS_PASSES; P++) {
    a[P] = hess_pair(P) / 32;
    b[P] = hess_pair(P) % 32;
    in_last[P] = hess_pass_in_knot(true, P);
  }
  return HESS_PASSES;
}

// Every pass of the table that runs in this knot class, with its row-group mask, contracted with lam over all rows the
// pass evaluates: H[p * NIN + q] receives the block entry of local inputs p = 3a + i <= q = 3b + j (the upper triangle
// of a diagonal block), cnt[p * NIN + q] counts how often each entry was written.
struct PassSink {
  const double* lam;
  double acc[3][3];
  void operator()(int, double) {}
  void operator()(int rho, const Dual2& d) {
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) acc[i][j] += lam[rho] * d.h[i][j];
  }
};
template <bool LAST, int P>
static void run_pass(const double* x, double h, const Params& pr, const double* lam, double* H, int* cnt) {
  if constexpr (hess_pass_in_knot(LAST, P)) {
    PassSink s{lam, {}};
    hess_pass<LAST, P>(x, h, pr, s);
    constexpr int a = HessPassOf<P>::a, b = HessPassOf<P>::b;
    for (int i = 0; i < 3; i++)
      for (int j = (a == b ? i : 0); j < 3; j++) {
        H[(3 * a + i) * NIN + 3 * b + j] = s.acc[i][j];
        cnt[(3 * a + i) * NIN + 3 * b + j] += 1;
      }
  }
}
template <bool LAST, int... P>
static void run_passes(const double* x, double h, const Params& pr, const double* lam, double* H, int* cnt,
                       std::integer_sequence<int, P...>) {
  (run_pass<LAST, P>(x, h, pr, lam, H, cnt), ...);
}

extern "C" int kino_hess_host_passes(int last, const double* in, double h, const double* prm, const double* lam,
                                     double* H, int* cnt) {
  const Params pr{prm[0], prm[1], {prm[2], prm[3], prm[4]}, {prm[5], prm[6], prm[7]}};  // mu, mass, Ib, Ib_inv
  double x[NIN];
  for (int i = 0; i < NIN; i++) x[i] = (last && i >= 60) ? 0.0 : in[i];
  if (last) run_passes<true>(x, h, pr, lam, H, cnt, std::make_integer_sequence<int, HESS_PASSES>{});
  else run_passes<false>(x, h, pr, lam, H, cnt, std::make_integer_sequence<int, HESS_PASSES>{});
  return 0;
}
