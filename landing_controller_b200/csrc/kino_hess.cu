// kino_hess.cu -- batched Lagrangian Hessian of the kino-dynamic ("full-body") landing NLP (SURVEY 8 f-2):
// H = d2/dx2 (lam_f f(x) + lam_g' g(x)) with g the constraint function of kino.cu and f the terminal cost of k_kino_cost,
// the upper triangle in CasADi CCS order (the convention of nlp_hess_l).  Exact forward-over-forward derivatives of the
// same knot function (kino_knot.cuh, Dual2): one pass per pair of input triples whose cross block is non-zero
// (kino::hess_pair), one thread per (scenario, knot, pass).  A thread contracts the second-order part of every row with
// lam_g in registers and writes its 3 x 3 block to the CCS positions of a host-made table: every entry of the pattern has
// exactly one writer (the plan checks it), so there are no atomics, and every entry is written on every call.
#include <algorithm>
#include <random>
#include <vector>

#include "kernels.cuh"
#include "kino_knot.cuh"

namespace srb {
namespace {

using kino::Dual2;
using kino::HESS_PASSES;
using kino::NIN;
using kino::ROWS_INT;
constexpr int HESS_ROW_WORDS = (ROWS_INT + 31) / 32;

// Sink of a Hessian pass: a row typed double depends on neither triple; a Dual2 row with a second-order part in this
// block (host-made row mask) adds lam_g[row] * h to the block.  lam_g is read for those rows only.
struct HSink {
  CView lam;
  long long b, base;
  const unsigned* rows;
  double acc[3][3];
  __device__ __forceinline__ void operator()(int, double) {}
  __device__ __forceinline__ void operator()(int rho, const Dual2& v) {
    if (!((__ldg(rows + (rho >> 5)) >> (rho & 31)) & 1u)) return;
    const double l = lam.get(base + rho, b);
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
      for (int j = 0; j < 3; j++) acc[i][j] = fma(l, v.h[i][j], acc[i][j]);
  }
};

template <bool LAST, int P>
__device__ __forceinline__ void kino_hess_pass(const KinoHessArgs& a, long long b, int k) {
  double x[NIN];  // (loads of inputs the pass never uses are dead code)
#pragma unroll
  for (int v = 0; v < NIN; v++) x[v] = (LAST && v >= 60) ? 0.0 : a.x.get(kino_col(a.N, k, v), b);
  HSink s{a.lam_g, b, 48 + (long long)ROWS_INT * k, a.rows + ((LAST ? HESS_PASSES : 0) + P) * HESS_ROW_WORDS, {}};
  kino::hess_pass<LAST, P>(x, __ldg(a.dtv + k), a.pr, s);
  const int* pos = a.hpos + ((long long)k * HESS_PASSES + P) * 9;
#pragma unroll
  for (int ij = 0; ij < 9; ij++) {
    const int p = __ldg(pos + ij);
    if (p >= 0) a.hess.at(p, b) = s.acc[ij / 3][ij % 3];
  }
}
template <bool LAST, int P, int P1>
__device__ __forceinline__ void kino_hess_dispatch(const KinoHessArgs& a, long long b, int k, int g) {
  if constexpr (P < P1) {
    if (g == P) {
      if constexpr (kino::hess_pass_in_knot(LAST, P)) kino_hess_pass<LAST, P>(a, b, k);
    } else {
      kino_hess_dispatch<LAST, P + 1, P1>(a, b, k, g);
    }
  }
}

// Passes P0..P1-1; blockIdx.x = pass + (P1 - P0) * scenario block, so the passes of one (scenario block, knot) read the
// same x and lam_g and are scheduled together, as in k_kino_jac.  One kernel per class of passes (launch_kino_hess), so
// that the light pairs are not held to the register count of the rpy pairs.  The thread of (last knot, pass 0) also
// writes the terminal-cost diagonal 2 lam_f QN.
template <int P0, int P1>
__global__ void __launch_bounds__(128) k_kino_hess(KinoHessArgs a) {
  constexpr int NPASS = P1 - P0;
  const int g = P0 + (int)(blockIdx.x % NPASS);
  const long long b = (long long)(blockIdx.x / NPASS) * 128 + threadIdx.x;
  if (b >= a.B) return;
  const int N = a.N, k = blockIdx.y;  // (block-uniform dispatch)
  if (k == N - 2) kino_hess_dispatch<true, P0, P1>(a, b, k, g);
  else kino_hess_dispatch<false, P0, P1>(a, b, k, g);
  if (P0 == 0 && k == N - 2 && g == 0) {
    const double lf2 = 2.0 * a.lam_f.get(0, b);
#pragma unroll
    for (int i = 0; i < 12; i++) a.hess.at(__ldg(a.cpos + i), b) = lf2 * a.QN[i];
  }
}

}  // namespace

// ---------------------------------------------------------------- host: pattern, writers, row masks
KinoHessPlan make_kino_hess_plan(int N) {
  KinoHessPlan pl;
  pl.N = N;
  pl.nx = 12LL * N + 36LL * (N - 1);
  const int K = N - 1;
  // Exact knot-local structure: every ordered triple pair (a <= b), all inputs Dual2 with run-time seeds, at random
  // points, both knot classes.  nz[cls][a][b][3 i + j]: d2 L / dz_{3a+i} dz_{3b+j} can be non-zero; dep: the rows that
  // contribute to the block.
  std::mt19937_64 rng(12345);
  std::uniform_real_distribution<double> U(-1.0, 1.0);
  kino::Params pr{0.75, 8.252, {0.0576, 0.234, 0.28}, {17.4, 4.27, 3.58}};
  constexpr int T = NIN / 3;
  std::vector<char> nz((size_t)2 * T * T * 9, 0), dep((size_t)2 * T * T * ROWS_INT, 0);
  auto at = [&](int cls, int a, int b) { return ((size_t)cls * T + a) * T + b; };
  for (int cls = 0; cls < 2; cls++) {
    const bool last = cls == 1;
    for (int rep = 0; rep < 3; rep++) {
      double xv[NIN];
      for (int i = 0; i < NIN; i++) xv[i] = U(rng);
      for (int a = 0; a < T; a++)
        for (int b = a; b < T; b++) {
          if (last && b >= 20) continue;
          Dual2 in[NIN];
          for (int i = 0; i < NIN; i++) {
            in[i] = Dual2(xv[i]);
            if (i / 3 == a) in[i].a[i % 3] = 1.0;
            if (i / 3 == b) in[i].b[i % 3] = 1.0;
          }
          auto sink = [&](int rho, const Dual2& d) {
            for (int ij = 0; ij < 9; ij++)
              if (d.h[ij / 3][ij % 3] != 0.0) {
                nz[at(cls, a, b) * 9 + ij] = 1;
                dep[at(cls, a, b) * ROWS_INT + rho] = 1;
              }
          };
          kino::knot_rows<Dual2>(in, 0.03, pr, last, sink);
        }
    }
  }
  // the pair table must hold every non-zero block, once, in the knot classes it runs in
  std::vector<int> pass_of((size_t)T * T, -1);
  for (int P = 0; P < HESS_PASSES; P++) {
    const int a = kino::hess_pair(P) / 32, b = kino::hess_pair(P) % 32;
    if (a > b || b >= T || pass_of[(size_t)a * T + b] >= 0) { pl.err = "kino Hessian: malformed pair table"; return pl; }
    pass_of[(size_t)a * T + b] = P;
  }
  for (int cls = 0; cls < 2; cls++)
    for (int a = 0; a < T; a++)
      for (int b = a; b < T; b++) {
        bool any = false;
        for (int ij = 0; ij < 9; ij++) any = any || nz[at(cls, a, b) * 9 + ij];
        const int P = pass_of[(size_t)a * T + b];
        if (any && (P < 0 || !kino::hess_pass_in_knot(cls == 1, P))) {
          pl.err = "kino Hessian: the pair table misses the non-zero block of triples (" + std::to_string(a) + ", " +
                   std::to_string(b) + ")";
          return pl;
        }
      }
  pl.rows.assign((size_t)2 * HESS_PASSES * HESS_ROW_WORDS, 0u);
  for (int cls = 0; cls < 2; cls++)
    for (int P = 0; P < HESS_PASSES; P++) {
      const int a = kino::hess_pair(P) / 32, b = kino::hess_pair(P) % 32;
      for (int rho = 0; rho < ROWS_INT; rho++)
        if (dep[at(cls, a, b) * ROWS_INT + rho]) pl.rows[((size_t)cls * HESS_PASSES + P) * HESS_ROW_WORDS + rho / 32] |= 1u << (rho % 32);
    }
  // global entries (col, row), row <= col, with their writers -> CCS order
  struct E { long long col, row; int k, p, ij; };
  std::vector<E> ent;
  for (int k = 0; k < K; k++) {
    const int cls = k == K - 1;
    for (int P = 0; P < HESS_PASSES; P++) {
      if (!kino::hess_pass_in_knot(cls == 1, P)) continue;
      const int a = kino::hess_pair(P) / 32, b = kino::hess_pair(P) % 32;
      for (int ij = 0; ij < 9; ij++) {
        const int i = ij / 3, j = ij % 3;
        if (!nz[at(cls, a, b) * 9 + ij] || (a == b && i > j)) continue;  // (a diagonal block: its upper triangle)
        const long long ci = kino_col(N, k, 3 * a + i), cj = kino_col(N, k, 3 * b + j);
        ent.push_back({std::max(ci, cj), std::min(ci, cj), k, P, ij});
      }
    }
  }
  for (int i = 0; i < 12; i++) ent.push_back({12LL * (N - 1) + i, 12LL * (N - 1) + i, -1, 0, i});
  std::sort(ent.begin(), ent.end(), [](const E& a, const E& b) { return a.col != b.col ? a.col < b.col : a.row < b.row; });
  for (size_t p = 1; p < ent.size(); p++)
    if (ent[p].col == ent[p - 1].col && ent[p].row == ent[p - 1].row) {
      pl.err = "kino Hessian: entry (" + std::to_string(ent[p].row) + ", " + std::to_string(ent[p].col) + ") has two writers";
      return pl;
    }
  pl.nnz = (long long)ent.size();
  pl.sparsity.assign(2 + pl.nx + 1 + pl.nnz, 0);
  pl.sparsity[0] = pl.nx; pl.sparsity[1] = pl.nx;
  pl.hpos.assign((size_t)K * HESS_PASSES * 9, -1);
  pl.cpos.assign(12, 0);
  for (long long p = 0; p < pl.nnz; p++) {
    const E& e = ent[p];
    pl.sparsity[2 + e.col + 1] += 1;
    pl.sparsity[2 + pl.nx + 1 + p] = e.row;
    if (e.k < 0) pl.cpos[e.ij] = (int)p;
    else pl.hpos[((size_t)e.k * HESS_PASSES + e.p) * 9 + e.ij] = (int)p;
  }
  for (long long c = 0; c < pl.nx; c++) pl.sparsity[2 + c + 1] += pl.sparsity[2 + c];
  return pl;
}

int launch_kino_hess(const KinoHessArgs& a, cudaStream_t st) {
  const unsigned gx = (unsigned)((a.B + 127) / 128);
  constexpr int R = kino::HESS_RPY_END, J = kino::HESS_JPOS_END;
  k_kino_hess<0, R><<<dim3(gx * R, a.N - 1, 1), 128, 0, st>>>(a);                            // pairs with rpy
  k_kino_hess<R, J><<<dim3(gx * (J - R), a.N - 1, 1), 128, 0, st>>>(a);                      // joint-angle pairs
  k_kino_hess<J, HESS_PASSES><<<dim3(gx * (HESS_PASSES - J), a.N - 1, 1), 128, 0, st>>>(a);  // the rest
  return 3;
}

}  // namespace srb
