// tests/hostcheck/kino_host.cpp -- TEST HARNESS (CPU): compiles the product's kino-dynamic knot template
// (landing_controller_b200/csrc/kino_knot.cuh) for the host, so that the knot math and the pass table of the Jacobian
// kernels (kino::PassOf, kino::jac_pass) can be checked against the oracle without a GPU.  Not part of the product
// library and never used as a fallback.
#include <utility>

#include "../../landing_controller_b200/csrc/kino_knot.cuh"

using namespace srb::kino;

static Params params(const double* prm) {  // mu, mass, Ib[3], Ib_inv[3]
  return Params{prm[0], prm[1], {prm[2], prm[3], prm[4]}, {prm[5], prm[6], prm[7]}};
}

// Rows g[rho] of one knot and its full Jacobian jac[rho * NIN + v] by one Dual1 evaluation per input (the last knot has
// no inputs 60..71); entries of rows that do not depend on an input are left as the caller set them.
extern "C" int kino_host_knot(int last, const double* in, double h, const double* prm, double* g, double* jac) {
  const Params pr = params(prm);
  for (int v = 0; v < (last ? 60 : NIN); v++) {
    Dual1 z[NIN];
    for (int i = 0; i < NIN; i++) z[i] = Dual1(in[i], i == v ? 1.0 : 0.0);
    auto sink = [&](int rho, const Dual1& d) {
      g[rho] = d.v;
      jac[rho * NIN + v] = d.d[0];
    };
    knot_rows<Dual1>(z, h, pr, last != 0, sink);
  }
  return 0;
}

// The Jacobian as the kernels assemble it: every pass of the table that runs in this knot class, with its mask.
// jac[rho * NIN + v] receives what the passes emit; cnt[rho * NIN + v] counts how often each entry was emitted.
struct PassSink {
  double* jac;
  int* cnt;
  int v0;
  void operator()(int, double) const {}
  void operator()(int rho, const DualN<3>& d) const {
    for (int j = 0; j < 3; j++) {
      jac[rho * NIN + v0 + j] = d.d[j];
      cnt[rho * NIN + v0 + j] += 1;
    }
  }
};
template <bool LAST, int G>
static void run_pass(const double* x, double h, const Params& pr, double* jac, int* cnt) {
  if constexpr (pass_in_knot(LAST, G)) {
    PassSink s{jac, cnt, PassOf<G>::v0};
    jac_pass<LAST, G>(x, h, pr, s);
  }
}
template <bool LAST, int... G>
static void run_passes(const double* x, double h, const Params& pr, double* jac, int* cnt, std::integer_sequence<int, G...>) {
  (run_pass<LAST, G>(x, h, pr, jac, cnt), ...);
}

extern "C" int kino_host_passes(int last, const double* in, double h, const double* prm, double* jac, int* cnt) {
  const Params pr = params(prm);
  double x[NIN];
  for (int i = 0; i < NIN; i++) x[i] = (last && i >= 60) ? 0.0 : in[i];
  if (last) run_passes<true>(x, h, pr, jac, cnt, std::make_integer_sequence<int, JAC_PASSES>{});
  else run_passes<false>(x, h, pr, jac, cnt, std::make_integer_sequence<int, JAC_PASSES>{});
  return 0;
}
