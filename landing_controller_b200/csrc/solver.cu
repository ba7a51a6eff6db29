// solver.cu -- batched primal-dual interior-point solver for the SRB landing NLP (sm_100a, FP64).
//
// Replaces, for a whole batch of drop conditions, what the reference does one scenario at a time
// through CasADi's Nlpsol + IPOPT (nlpsol.cpp:555-635 -> IpoptInterface::solve; option set
// generate_landingCtrller_IPOPT.m:232-263; callers main_scripts/landing_optimization.m:305-311,
// generate_data/generate_training_data_automated.m:130-136).
//
// B200 design (device code in solver_dev.cuh)
//  * ONE persistent kernel; ONE CTA of 256 threads = ONE SCENARIO for the whole solve (all
//    interior-point iterations, line searches and inertia corrections run on the device, no host
//    round trip, no lock-step between scenarios); 2 CTAs resident per SM pull scenario ids from an
//    atomic work queue (longest expected first, k_order), so a slow scenario never stalls the others
//    and the latency-bound Cholesky chain of one scenario overlaps with the phases of its neighbour.
//  * Evaluation: one THREAD per knot (srb_knot.cuh), Jacobian and Hessian lists on different warps.
//  * Linear algebra: slacks and bound multipliers are eliminated; the remaining equality-constrained
//    QP (linearised Euler dynamics) is solved by a Riccati recursion with state (X_k, c_k) [24] and
//    control (f_k, c_{k+1}) [24].  Each stage is built in shared memory from the stage's entry
//    lists by a host-made "condensing schedule" (no atomics, deterministic), factored by a blocked
//    partial Cholesky (diagonal blocks in the registers of the two panel warps), and only the factors
//    needed by the forward sweep are written to the per-CTA scratch.
//  * Reductions (errors, step lengths, merit function) are shuffle + shared-memory block
//    reductions: every thread ends up with the identical value, so all control flow is
//    block-uniform and deterministic.
//
// The algorithm mirrors oracle/ip_ref.c step by step (that file is the CPU restatement used only
// by the tests and the CPU baseline).  There is no CPU path in this library.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "solver.cuh"
#include "srb_knot.cuh"
#include "solver_dev.cuh"

namespace srb {

namespace {

// ---------------------------------------------------------------- host: tables
struct HostTables {
  std::vector<int> all;
  size_t o_jl, o_hl, o_rptr, o_rterms, o_cptr, o_cterms, o_sm, o_tinit;
  std::vector<int> sm;  // shared-memory tables
  int o_g, n_g, o_qptr, o_qterms, o_uabh, o_uptr, o_uterms, n_u, s_rptr, s_rterms, s_cptr, s_cterms;
};

int sidx_host(int v) { return v < 36 ? v : (v >= 48 ? v - 12 : -1); }
int dyn_state_host(int rho) { return rho < 6 ? rho : (rho < 9 ? rho + 3 : rho - 3); }
int rowmap_last_host(int r) {
  if (r < 16) return r;
  if (r < 40) { const int l = (r - 16) / 6, j = (r - 16) % 6; return 16 + 12 * l + (j < 2 ? j : j + 6); }
  return r + 24;
}

HostTables build_tables_host() {
  Knot z{};
  z.h = 0.03; z.mu = 1; z.mass = 1;
  for (int i = 0; i < 3; i++) { z.Ib[i] = 1; z.Ibinv[i] = 1; }
  PatternSink pi, pl;
  NoLam nl;
  knot_eval<false, false, true, true>(z, pi, nl);
  knot_eval<true, false, true, true>(z, pl, nl);
  HostTables T;
  auto push = [&](const std::vector<int>& v) { size_t o = T.all.size(); T.all.insert(T.all.end(), v.begin(), v.end()); return o; };
  // last-knot emission index -> interior emission index
  std::vector<int> jl(NJ_LAST), hl(NH_LAST);
  for (int e = 0; e < NJ_LAST; e++) {
    const int row = rowmap_last_host(pl.jac[e].first), var = pl.jac[e].second;
    int f = -1;
    for (int q = 0; q < NJ_INT; q++) if (pi.jac[q].first == row && pi.jac[q].second == var) f = q;
    jl[e] = f;
  }
  for (int e = 0; e < NH_LAST; e++) {
    int f = -1;
    for (int q = 0; q < NH_INT; q++) if (pi.hes[q] == pl.hes[e]) f = q;
    hl[e] = f;
  }
  T.o_jl = push(jl);
  T.o_hl = push(hl);
  auto pushs = [&](const std::vector<int>& v) { int o = (int)T.sm.size(); T.sm.insert(T.sm.end(), v.begin(), v.end()); return o; };
  const int NULL_E = NJ_INT;  // padding slot of the list (always 0.0): a term that adds nothing
  // dynamics entries -> G
  std::vector<int> gp;
  for (int e = 0; e < NJ_INT; e++)
    if (pi.jac[e].first < 12 && pi.jac[e].second < 36)
      gp.push_back(e | ((dyn_state_host(pi.jac[e].first) * 36 + pi.jac[e].second) << 10));
  T.n_g = (int)gp.size();
  T.o_g = pushs(gp);
  // unified condensing targets: lower triangle in elimination order; Hessian entry + sigma-weighted terms.
  // The term lists are padded with null terms (the padding slot of the J list is 0.0) to pairs (condensing) or fours
  // (row / column schedules): the device loops run two / four terms per trip, so their dependent loads overlap
  auto rot = [](int s) { return s < 24 ? s + 24 : s - 24; };
  std::map<int, std::vector<int>> tg;
  std::map<int, int> th;
  for (int e = 0; e < NH_INT; e++) {
    int a = rot(sidx_host(pi.hes[e].first)), b2 = rot(sidx_host(pi.hes[e].second));
    if (a < b2) std::swap(a, b2);
    if (th.count(a * NW + b2)) { fprintf(stderr, "landing: duplicate Hessian target\n"); abort(); }
    th[a * NW + b2] = e;
    tg[a * NW + b2];
  }
  std::vector<std::vector<int>> rows(RK);
  for (int e = 0; e < NJ_INT; e++) rows[pi.jac[e].first].push_back(e);
  for (int rho = 12; rho < RK; rho++)
    for (size_t a = 0; a < rows[rho].size(); a++)
      for (size_t b2 = a; b2 < rows[rho].size(); b2++) {
        const int ea = rows[rho][a], eb = rows[rho][b2];
        int i = rot(sidx_host(pi.jac[ea].second)), j = rot(sidx_host(pi.jac[eb].second));
        if (i < j) std::swap(i, j);
        tg[i * NW + j].push_back((rho << 20) | (ea << 10) | eb);
        if (i == j && ea != eb) tg[i * NW + j].push_back((rho << 20) | (eb << 10) | ea);
      }
  for (int m = 0; m < NW; m++)
    if (!tg.count(m * NW + m)) { fprintf(stderr, "landing: stage diagonal %d is not a condensing target\n", m); abort(); }
  // deal targets to threads longest-first for balance; term lists padded to pairs with null terms
  std::vector<std::pair<int, int>> order;
  for (auto& kv : tg) order.push_back({-(int)kv.second.size(), kv.first});
  std::sort(order.begin(), order.end());
  std::vector<int> uptr{0}, uabh, uterms;
  for (auto& o : order) {
    uabh.push_back(o.second | ((th.count(o.second) ? th[o.second] + 1 : 0) << 12));
    for (int t : tg[o.second]) uterms.push_back(t);
    if (uterms.size() & 1) uterms.push_back((NULL_E << 10) | NULL_E);
    uptr.push_back((int)uterms.size());
  }
  T.n_u = (int)uabh.size();
  {
    // inverse of the target list for the accumulator tiles of the factorisation (sweeps.cuh: backward_stages, S3)
    std::map<int, int> pos;
    for (int i = 0; i < (int)uabh.size(); i++) pos[uabh[i] & 4095] = i;
    std::vector<int> tinit(NTILE * 32);
    for (int tile = 0; tile < NTILE; tile++)
      for (int lane = 0; lane < 32; lane++) {
        const int I = tile_I(tile), J = tile_J(tile), g = lane >> 2, t = lane & 3;
        unsigned word = 0;
        for (int e = 0; e < 2; e++) {
          const int row = 8 * I + g, col = 8 * J + 2 * t + e;
          unsigned idx = 0xffffu;
          if (I == 6) { if (g == 0) idx = (unsigned)(CT_Q + col); }
          else if (col <= row && pos.count(row * NW + col)) idx = (unsigned)pos[row * NW + col];
          word |= idx << (16 * e);
        }
        tinit[tile * 32 + lane] = (int)word;
      }
    T.o_tinit = push(tinit);
  }
  T.o_uabh = pushs(uabh);
  T.o_uptr = pushs(uptr);
  T.o_uterms = pushs(uterms);
  // stage gradient: per stage variable in elimination order
  std::vector<int> qptr{0}, qterms;
  for (int m = 0; m < NW; m++) {
    for (int e = 0; e < NJ_INT; e++)
      if (pi.jac[e].first >= 12 && sidx_host(pi.jac[e].second) >= 0 && rot(sidx_host(pi.jac[e].second)) == m)
        qterms.push_back((pi.jac[e].first << 10) | e);
    if (qterms.size() & 1) qterms.push_back(NULL_E);
    qptr.push_back((int)qterms.size());
  }
  T.o_qptr = pushs(qptr);
  T.o_qterms = pushs(qterms);
  // row schedule: per row, (stage var, e)
  std::vector<int> rptr(RK + 1, 0), rterms;
  for (int rho = 0; rho < RK; rho++) {
    if (rho >= 12)
      for (int e : rows[rho]) rterms.push_back((sidx_host(pi.jac[e].second) << 10) | e);
    while (rterms.size() & 3) rterms.push_back(NULL_E);  // (stage variable 0, zero list slot)
    rptr[rho + 1] = (int)rterms.size();
  }
  T.o_rptr = push(rptr);
  T.o_rterms = push(rterms);
  T.s_rptr = pushs(rptr);
  T.s_rterms = pushs(rterms);
  // column schedule: per local variable (60), (rho, e)
  std::vector<int> cptr{0}, cterms;
  for (int v = 0; v < 60; v++) {
    for (int e = 0; e < NJ_INT; e++)
      if (pi.jac[e].second == v) cterms.push_back((pi.jac[e].first << 10) | e);
    while (cterms.size() & 3) cterms.push_back(NULL_E);  // (row 0, zero list slot)
    cptr.push_back((int)cterms.size());
  }
  T.o_cptr = push(cptr);
  T.o_cterms = push(cterms);
  T.s_cptr = pushs(cptr);
  T.s_cterms = pushs(cterms);
  T.o_sm = push(T.sm);
  return T;
}

}  // namespace

#define CUS(call)                                                            \
  do {                                                                       \
    cudaError_t e_ = (call);                                                 \
    if (e_ != cudaSuccess) {                                                 \
      *err = std::string(#call) + ": " + cudaGetErrorString(e_);             \
      return LANDING_ERR_CUDA;                                               \
    }                                                                        \
  } while (0)

// ---------------------------------------------------------------- work-queue order (longest expected first)
// The scenarios of a sweep need 40 ... 300 interior-point iterations each; with ~300 scenarios in flight the sweep ends
// when the last long one does, so the queue hands out the scenarios with the largest drop energy g z0 + |v0|^2 / 2
// first (they tend to need more iterations: correlation 0.2 ... 0.45 on the grid and random sweeps; a late long scenario
// otherwise leaves the GPU nearly idle for its whole solve).  Rank by counting (O(B^2) comparisons, shared-memory tiles).
namespace {
__global__ void __launch_bounds__(256) k_order(const double* __restrict__ drops, long long B, int* __restrict__ order) {
  __shared__ double tile[256];
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  auto key = [&](long long b) {
    const double* d = drops + 12 * b;
    const double k = 9.81 * d[2] + 0.5 * (d[9] * d[9] + d[10] * d[10] + d[11] * d[11]);
    return k == k ? k : HUGE_VAL;  // NaN input: first in the queue (total order, so the ranks are a permutation)
  };
  const double mine = i < B ? key(i) : 0.0;
  long long rank = 0;
  for (long long j0 = 0; j0 < B; j0 += 256) {
    const long long j = j0 + threadIdx.x;
    __syncthreads();
    tile[threadIdx.x] = j < B ? key(j) : -HUGE_VAL;
    __syncthreads();
    const int n = (int)(B - j0 < 256 ? B - j0 : 256);
    for (int t = 0; t < n; t++) {
      const double o = tile[t];
      rank += (o > mine || (o == mine && j0 + t < i)) ? 1 : 0;
    }
  }
  if (i < B) order[rank] = (int)i;
}
// large sweeps: the same order (key descending, ties in input order) from a stable radix sort instead of O(B^2) counting
__global__ void __launch_bounds__(256) k_order_keys(const double* __restrict__ drops, long long B, double* __restrict__ keys,
                                                    int* __restrict__ ids) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= B) return;
  const double* d = drops + 12 * i;
  const double k = 9.81 * d[2] + 0.5 * (d[9] * d[9] + d[10] * d[10] + d[11] * d[11]);
  keys[i] = k == k ? k : HUGE_VAL;
  ids[i] = (int)i;
}
}  // namespace

// ---------------------------------------------------------------- FP64 FMA peak (measured, for the roofline)
namespace {
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters) {
  // 16 independent DFMA chains per thread; 8 warps x 8 CTAs per SM keep the FP64 pipe full
  double a[16];
#pragma unroll
  for (int i = 0; i < 16; i++) a[i] = 1.0 + 1e-9 * (threadIdx.x + i);
  const double m = 1.0000001, c = 1e-9;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 16; i++) a[i] = fma(a[i], m, c);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) s += a[i];
  if (s == 123.456) out[0] = s;  // never true; keeps the chains alive
}
}  // namespace

int fp64_peak_run(cudaStream_t st, double* tflops, std::string* err) {
  int dev = 0, n_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  double* d_out = nullptr;
  CUS(cudaMalloc(&d_out, 8));
  cudaEvent_t e0, e1;
  CUS(cudaEventCreate(&e0));
  CUS(cudaEventCreate(&e1));
  const int grid = n_sm * 8, iters = 20000;
  double best = 0;
  for (int rep = 0; rep < 4; rep++) {
    CUS(cudaEventRecord(e0, st));
    k_fp64_peak<<<grid, 256, 0, st>>>(d_out, iters);
    CUS(cudaEventRecord(e1, st));
    CUS(cudaEventSynchronize(e1));
    float ms = 0;
    CUS(cudaEventElapsedTime(&ms, e0, e1));
    const double tf = 2.0 * 16.0 * iters * 256.0 * grid / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d_out);
  *tflops = best;
  return LANDING_OK;
}

void solver_free(SolverWorkspace& ws) {
  if (ws.counter) cudaFree(ws.counter);
  if (ws.zeros) cudaFree(ws.zeros);
  if (ws.kt) cudaFree(ws.kt);
  if (ws.tab.dev) cudaFree(ws.tab.dev);
  ws.counter = nullptr;
  ws.zeros = nullptr;
  ws.kt = nullptr;
  ws.tab = SolverTables{};
  ws.ready = false;
}

int solver_run(SolverWorkspace& ws, const DevicePlan& pl, long long B,
               const landing_problem& pb, const double* dtv, const unsigned char* csm, const landing_options& opt,
               const landing_solve_io& io, cudaStream_t st, int* launches, std::string* err) {
  const int N = pl.N;
  if (N - 1 > 1023 / 1) { *err = "landing_solve_batch: N too large"; return LANDING_ERR_ARG; }
  if (!io.x_star || !io.f_star || !io.status || !io.iters) {
    *err = "landing_solve_batch: x_star, f_star, status and iters are required";
    return LANDING_ERR_ARG;
  }
  if (!ws.ready) {
    solver_free(ws);  // (a previous attempt may have failed half way)
    HostTables T = build_tables_host();
    CUS(cudaMalloc(&ws.tab.dev, sizeof(int) * T.all.size()));
    CUS(cudaMemcpy(ws.tab.dev, T.all.data(), sizeof(int) * T.all.size(), cudaMemcpyHostToDevice));
    const int* d = ws.tab.dev;
    ws.tab.jl_last = d + T.o_jl; ws.tab.hl_last = d + T.o_hl;
    ws.tab.r_ptr = d + T.o_rptr; ws.tab.r_terms = d + T.o_rterms;
    ws.tab.c_ptr = d + T.o_cptr; ws.tab.c_terms = d + T.o_cterms;
    ws.tab.sm_src = d + T.o_sm; ws.tab.sm_count = (int)T.sm.size();
    ws.tab.tinit = d + T.o_tinit;
    if (ws.tab.sm_count > TBL_INTS) { *err = "landing_solve_batch: shared-memory tables exceed their region"; return LANDING_ERR_ARG; }
    ws.tab.o_g = T.o_g; ws.tab.n_g = T.n_g; ws.tab.o_qptr = T.o_qptr; ws.tab.o_qterms = T.o_qterms;
    ws.tab.o_uabh = T.o_uabh; ws.tab.o_uptr = T.o_uptr; ws.tab.o_uterms = T.o_uterms; ws.tab.n_u = T.n_u;
    ws.tab.o_rptr = T.s_rptr; ws.tab.o_rterms = T.s_rterms; ws.tab.o_cptr = T.s_cptr; ws.tab.o_cterms = T.s_cterms;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&ws.n_sm, cudaDevAttrMultiProcessorCount, dev);
    CUS(cudaMalloc(&ws.counter, sizeof(int)));
    CUS(cudaMalloc(&ws.kt, KT_BYTES));
    CUS(cudaMalloc(&ws.zeros, sizeof(double) * 16));
    CUS(cudaMemset(ws.zeros, 0, sizeof(double) * 16));
    CUS(cudaFuncSetAttribute(k_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SM_TOTAL * sizeof(double))));
    if (const char* e = getenv("LANDING_CARVEOUT"))  // experiments: shared-memory carve-out in percent
      CUS(cudaFuncSetAttribute(k_solve, cudaFuncAttributePreferredSharedMemoryCarveout, atoi(e)));
    ws.ready = true;  // only now: a failure above leaves the workspace to be set up again by the next call
  }
  const long long slot = slot_doubles(N);
  const long long nslots = (long long)ws.n_sm * CTAS_PER_SM;
  CUS(ws.scratch.reserve(sizeof(double) * slot * nslots));
  const long long m = pl.m;
  KParams P{};
  P.N = N; P.K = N - 1; P.nx = pl.nx; P.MR = 36 + RK * (N - 1);
  P.B = B; P.pb = pb; P.pb.dt = nullptr; P.pb.cs = nullptr; P.dtv = dtv; P.csm = csm; P.opt = opt;
  P.run_qx = 0;
  for (int i = 0; i < 12; i++) P.run_qx |= (pb.QX[i] != 0.0);
  P.opt.reserved[0] = pl.m;  // m, for the dual scaling s_d
  P.zeros = ws.zeros;
  P.counter = ws.counter; P.scratch = ws.scratch.as<double>(); P.slot = slot; P.tab = ws.tab; P.kt = ws.kt;
  P.drops = io.drops; P.x0 = io.x0; P.x_star = io.x_star; P.f_star = io.f_star; P.lam_g = io.lam_g;
  P.viol = io.viol; P.status = io.status; P.iters = io.iters;
#ifdef SRB_PROF
  static const bool want_prof = getenv("LANDING_PROF") != nullptr;
#else
  static const bool want_prof = false;
#endif
  unsigned long long* d_prof = nullptr;
  if (want_prof) {
    CUS(cudaMalloc(&d_prof, sizeof(unsigned long long) * PH_COUNT));
    CUS(cudaMemsetAsync(d_prof, 0, sizeof(unsigned long long) * PH_COUNT, st));
  }
  P.prof = d_prof;
  CUS(cudaMemsetAsync(ws.counter, 0, sizeof(int), st));
  static const bool fifo = getenv("LANDING_FIFO") != nullptr;  // experiments: hand the scenarios out in input order
  if (!fifo && B > 1 && B < (1LL << 31)) {
    const bool by_sort = B > 16384;  // (rank by counting is O(B^2): 25 us at 1k, 0.4 ms at 16k; a radix sort beyond)
    size_t sort_bytes = 0;
    if (by_sort)
      CUS(cub::DeviceRadixSort::SortPairsDescending(nullptr, sort_bytes, (const double*)nullptr, (double*)nullptr,
                                                    (const int*)nullptr, (int*)nullptr, (int)B, 0, 64, st));
    CUS(ws.order.reserve(sizeof(int) * B + (by_sort ? (sizeof(double) * 2 + sizeof(int)) * B + sort_bytes + 512 : 0)));
    int* order = ws.order.as<int>();
    if (by_sort) {
      char* base = reinterpret_cast<char*>(order) + ((sizeof(int) * B + 255) / 256) * 256;
      double* k_in = reinterpret_cast<double*>(base);
      double* k_out = k_in + B;
      int* id_in = reinterpret_cast<int*>(k_out + B);
      void* tmp = reinterpret_cast<char*>(id_in) + ((sizeof(int) * B + 255) / 256) * 256;
      k_order_keys<<<(unsigned)((B + 255) / 256), 256, 0, st>>>(P.drops, B, k_in, id_in);
      CUS(cub::DeviceRadixSort::SortPairsDescending(tmp, sort_bytes, k_in, k_out, id_in, order, (int)B, 0, 64, st));
      *launches += 2;
    } else {
      k_order<<<(unsigned)((B + 255) / 256), 256, 0, st>>>(P.drops, B, order);
      *launches += 1;
    }
    P.order = order;
  }
  if (P.lam_g) CUS(cudaMemsetAsync(P.lam_g, 0, sizeof(double) * m * B, st));
  long long gcap = nslots;
  if (const char* e = getenv("LANDING_GRID")) gcap = std::max(1LL, std::min<long long>(nslots, atoll(e)));  // experiments
  const int grid = (int)std::min<long long>(gcap, B);
  k_kinds<<<1, 256, 0, st>>>(P);
  k_solve<<<grid, NT, SM_TOTAL * sizeof(double), st>>>(P);
  *launches += 2;
  CUS(cudaGetLastError());
  if (want_prof) {
    unsigned long long h[PH_COUNT];
    CUS(cudaStreamSynchronize(st));
    CUS(cudaMemcpy(h, d_prof, sizeof h, cudaMemcpyDeviceToHost));
    cudaFree(d_prof);
    static const char* names[] = {"eval", "row_errors", "dual_inf", "mu/yhat", "backward", "forward", "row_steps", "linesearch", "accept"};
    double tot = 0;
    for (int i = 0; i < PH_NBACK; i++) tot += (double)h[i];
    fprintf(stderr, "[landing prof] B=%lld iterations=%llu backward sweeps=%llu (%.2f per iteration), %.0f cycles per iteration\n",
            B, h[PH_NITER], h[PH_NBACK], (double)h[PH_NBACK] / (double)std::max(1ull, h[PH_NITER]), tot / (double)std::max(1ull, h[PH_NITER]));
    for (int i = 0; i < PH_NBACK; i++)
      fprintf(stderr, "[landing prof]   %-11s %6.1f%%  %9.0f cycles per iteration\n", names[i], 100.0 * (double)h[i] / tot,
              (double)h[i] / (double)std::max(1ull, h[PH_NITER]));
    static const char* bn[] = {"wait+sync", "P1 G,q", "P2 T=PG", "P3 tiles", "P4 targets", "(unused)", "P6 store", "", "P5 chol diag+panel", "P5 chol trailing"};
    for (int i = 0; i < 10; i++)
      if (bn[i][0] && i != 5)
        fprintf(stderr, "[landing prof]   backward %-18s %8.0f cycles per stage\n", bn[i],
                (double)h[PH_B_WAIT + i] / (double)std::max(1ull, h[PH_B_STAGES]));
    static const char* fn[] = {"wait+sync", "rhs,G", "L^-T solve", "next state"};
    const double fst = (double)std::max(1ull, h[PH_NITER]) * (P.K);
    for (int i = 0; i < 4; i++)
      fprintf(stderr, "[landing prof]   forward %-18s %8.0f cycles per stage\n", fn[i], (double)h[PH_F_WAIT + i] / fst);
    for (int i = 0; i < 8; i++)
      if (h[PH_X0 + i]) fprintf(stderr, "[landing prof]   X%d %10.0f cycles per iteration\n", i, (double)h[PH_X0 + i] / (double)std::max(1ull, h[PH_NITER]));
    fprintf(stderr, "[landing prof]   one lap of the instrumentation costs %.0f cycles\n",
            (double)h[PH_CAL] / (4.0 * (double)std::max(1ull, h[PH_NITER])));
  }
  return LANDING_OK;
}

}  // namespace srb
