// capi.cu -- the thin C-ABI layer of liblanding_b200.so (include/landing_b200.h).
// Host side only: context, device staging of host buffers, launches.  No CPU compute path:
// every entry point that produces numbers needs a CUDA device and fails loudly without one.
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "kernels.cuh"
#include "solver.cuh"

using namespace srb;

namespace {
thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(LANDING_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));      \
  } while (0)
// restores the calling thread's current device when an entry point returns
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev); else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
}  // namespace

struct landing_ctx {
  int N = 0, device = 0;
  std::shared_ptr<const HostPlan> plan;
  DevicePlan dpl{};
  cudaStream_t stream = nullptr;
  int* d_maps = nullptr;
  long long launches = 0;
  DeviceBuf stage;  // device staging of host-buffer calls (stage_in)
  MappedBuf pin;    // the same for small evaluation calls, zero-copy
  DeviceBuf tr;     // transposed (SoA) copies of AoS batches (aos_to_soa)
  SolverWorkspace ws;
  // knot spacings of the current call: pinned host staging + device copy (landing_problem.dt or uniform)
  PinnedBuf h_dt;
  DeviceBuf d_dt;
  // contact schedule of the current call (formulation 1): bit mask per knot
  PinnedBuf h_cs;
  DeviceBuf d_cs;
  // kino-dynamic NLP (landing_kino_eval_batch): host plan and its device tables, made on first use
  std::shared_ptr<const KinoPlan> kino;
  int* d_kino = nullptr;
  // its Lagrangian Hessian (landing_kino_hess_batch): pattern, writer and row-mask tables, made on first use
  std::shared_ptr<const KinoHessPlan> khess;
  int* d_khess = nullptr;
  // scratch of its KKT residuals (landing_kino_kkt_batch): g, and grad_x when the caller does not ask for it
  DeviceBuf kkt;
  // its interior-point Newton step (landing_kino_step_batch): plan tables + scenario counter, made on first use, and the
  // factor scratch of the resident CTAs
  std::shared_ptr<const KinoStepHost> kstep;
  int* d_kstep = nullptr;
  int kstep_grid = 0;
  DeviceBuf kstep_scr;
};

// dt[0..N-2] of this call on the device (stream-ordered): the caller's vector or the uniform T/(N-1)
static int stage_dt(landing_ctx* c, const double* dt, double T) {
  const int K = c->N - 1;
  CU(c->h_dt.reserve(sizeof(double) * K));
  CU(c->d_dt.reserve(sizeof(double) * K));
  CU(cudaStreamSynchronize(c->stream));  // the previous call's copies out of h_dt and h_cs (stage_cs) have completed
  for (int k = 0; k < K; k++) {
    const double h = dt ? dt[k] : T / (double)K;
    if (!(h > 0.0)) return fail(LANDING_ERR_ARG, "landing_problem: knot spacings must be positive");
    c->h_dt.as<double>()[k] = h;
  }
  CU(cudaMemcpyAsync(c->d_dt.as<double>(), c->h_dt.as<double>(), sizeof(double) * K, cudaMemcpyHostToDevice, c->stream));
  return LANDING_OK;
}

// the contact schedule of formulation 1 on the device (after stage_dt, whose synchronisation covers h_cs)
static int stage_cs(landing_ctx* c, const landing_problem* pb) {
  if (pb->formulation == 0) return LANDING_OK;
  if (pb->formulation != 1) return fail(LANDING_ERR_ARG, "landing_problem: formulation must be 0 or 1");
  if (!pb->cs) return fail(LANDING_ERR_ARG, "landing_problem: formulation 1 needs the contact schedule cs[4 (N-1)]");
  if (!(pb->delta_c > 0.0)) return fail(LANDING_ERR_ARG, "landing_problem: delta_c must be positive");
  const int K = c->N - 1;
  CU(c->h_cs.reserve(K));
  CU(c->d_cs.reserve(K));
  for (int k = 0; k < K; k++) {
    unsigned m = 0;
    for (int l = 0; l < 4; l++) m |= (pb->cs[4 * k + l] != 0) << l;
    c->h_cs.as<unsigned char>()[k] = (unsigned char)m;
  }
  CU(cudaMemcpyAsync(c->d_cs.as<unsigned char>(), c->h_cs.as<unsigned char>(), K, cudaMemcpyHostToDevice, c->stream));
  return LANDING_OK;
}

// One buffer argument of a batched call: `bytes` at the caller's input `in` or output `out` (both NULL: absent).
// `dev` is what the kernels read or write (stage_in); `aos` the caller-layout buffer while they use a transposed copy.
struct Piece {
  const void* in;
  void* out;
  size_t bytes;
  void* dev;
  void* aos;
  template <class T>
  T* at() const { return static_cast<T*>(dev); }
};
template <class T>
static Piece input(const T* p, long long n) { return {p, nullptr, sizeof(T) * n, nullptr, nullptr}; }
template <class T>
static Piece output(T* p, long long n) { return {nullptr, p, sizeof(T) * n, nullptr, nullptr}; }
static size_t padded(size_t bytes) { return (bytes + 7) & ~(size_t)7; }
static size_t staged_bytes(const Piece* pc, int n) {
  size_t tot = 256;
  for (int i = 0; i < n; i++)
    if (pc[i].in || pc[i].out) tot += padded(pc[i].bytes);
  return tot;
}

// Host buffers of a batched call.  LANDING_DEVICE: the kernels use the caller's pointers.  LANDING_HOST: the present
// pieces are laid out in the context's grow-only staging buffer and the inputs copied in (cudaMemcpyAsync on the
// context's stream); stage_out() copies the outputs back and synchronises the stream once.
// zero_copy (small host calls -- the CasADi ABI's one scenario per call above all): the pieces go to a mapped pinned
// buffer instead, the CPU copies the inputs in, the kernels read them and write their results through the device alias
// of that buffer, and the CPU copies the results out after the stream synchronisation: one launch + one synchronisation
// per call instead of up to a dozen pageable cudaMemcpyAsync.  Not for kernels that accumulate with device-scope atomics
// (nlp_grad's parameter sensitivities).
static int stage_in(landing_ctx* c, int memspace, Piece* pc, int n, bool zero_copy = false) {
  if (memspace != LANDING_HOST) {
    for (int i = 0; i < n; i++) pc[i].dev = pc[i].in ? const_cast<void*>(pc[i].in) : pc[i].out;
    return LANDING_OK;
  }
  if (zero_copy) CU(c->pin.reserve(staged_bytes(pc, n)));
  else CU(c->stage.reserve(staged_bytes(pc, n)));
  char* cur = zero_copy ? c->pin.as<char>() : c->stage.as<char>();
  for (int i = 0; i < n; i++) {
    pc[i].dev = nullptr;
    if (!pc[i].in && !pc[i].out) continue;
    pc[i].dev = cur;
    if (pc[i].in && zero_copy) std::memcpy(cur, pc[i].in, pc[i].bytes);
    else if (pc[i].in) CU(cudaMemcpyAsync(cur, pc[i].in, pc[i].bytes, cudaMemcpyHostToDevice, c->stream));
    cur += padded(pc[i].bytes);
  }
  return LANDING_OK;
}
static int stage_out(landing_ctx* c, int memspace, const Piece* pc, int n, bool zero_copy = false) {
  if (memspace != LANDING_HOST) return LANDING_OK;
  if (zero_copy) CU(cudaStreamSynchronize(c->stream));
  for (int i = 0; i < n; i++) {
    if (!pc[i].out) continue;
    if (zero_copy) std::memcpy(pc[i].out, pc[i].dev, pc[i].bytes);
    else CU(cudaMemcpyAsync(pc[i].out, pc[i].dev, pc[i].bytes, cudaMemcpyDeviceToHost, c->stream));
  }
  if (!zero_copy) CU(cudaStreamSynchronize(c->stream));
  return LANDING_OK;
}

// AoS batches (one CasADi vector per scenario) would make every warp access 32 different rows: for batches (B >= 64)
// the kernels run on transposed (SoA) copies instead and the results are transposed back through shared-memory tiles
// (3 x the traffic of a SoA call, but coalesced: DESIGN.md 2.2).  Small batches (the CasADi ABI: B = 1) go direct.
// pc[0..n) are staged [B][n_i] double arrays: the inputs are transposed into the context's scratch, the outputs
// redirected to it, and *layout becomes LANDING_SOA; soa_to_aos() transposes the outputs back after the launch.
static int aos_to_soa(landing_ctx* c, long long B, int* layout, Piece* pc, int n) {
  if (*layout != LANDING_AOS || B < 64) return LANDING_OK;
  CU(c->tr.reserve(staged_bytes(pc, n)));
  double* cur = c->tr.as<double>();
  for (int i = 0; i < n; i++) {
    if (!pc[i].dev) continue;
    const long long rows = (long long)(pc[i].bytes / sizeof(double)) / B;
    if (pc[i].in) c->launches += launch_transpose(pc[i].at<const double>(), cur, B, rows, c->stream);  // [B][n] -> [n][B]
    pc[i].aos = pc[i].dev;
    pc[i].dev = cur;
    cur += rows * B;
  }
  *layout = LANDING_SOA;
  return LANDING_OK;
}
static void soa_to_aos(landing_ctx* c, long long B, Piece* pc, int n) {
  for (int i = 0; i < n; i++)
    if (pc[i].out && pc[i].aos) {
      const long long rows = (long long)(pc[i].bytes / sizeof(double)) / B;
      // [n][B] -> [B][n]
      c->launches += launch_transpose(pc[i].at<const double>(), static_cast<double*>(pc[i].aos), rows, B, c->stream);
      pc[i].dev = pc[i].aos;
    }
}

extern "C" {

void landing_destroy(landing_ctx* c);

const char* landing_last_error(void) { return g_err.c_str(); }

int landing_dims_for(int N, long long d[6]) {
  if (N < 3 || !d) return fail(LANDING_ERR_ARG, "landing_dims_for: need N >= 3");
  d[0] = N;
  d[1] = 36LL * N - 24;
  d[2] = 13LL * N + 81;
  d[3] = 104LL * N - 92;
  d[4] = 385LL * N - 421;
  d[5] = 189LL * (N - 1);
  return LANDING_OK;
}

const long long* landing_sparsity_for(int N, int which) {
  if (N < 3) return nullptr;
  auto pl = get_plan(N);
  switch (which) {
    case 0: return pl->spJ.data();
    case 1: return pl->spH.data();
    case 2: return pl->spDense[0].data();  // x
    case 3: return pl->spDense[1].data();  // p
    case 4: return pl->spDense[2].data();  // scalar
    case 5: return pl->spDense[3].data();  // g / lam_g
    default: return nullptr;
  }
}

int landing_create(int N, int device, landing_ctx** out) {
  if (!out || N < 3) return fail(LANDING_ERR_ARG, "landing_create: need N >= 3 and a ctx pointer");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(LANDING_ERR_NOGPU, "landing_create: no CUDA device (this library has no CPU path)");
  if (device < 0 || device >= ndev) return fail(LANDING_ERR_ARG, "landing_create: bad device index");
  DeviceGuard guard_(device);
  landing_ctx* c = new landing_ctx();
  c->N = N;
  c->device = device;
  c->plan = get_plan(N);
  const HostPlan& pl = *c->plan;
  const size_t nj = pl.jmap.size(), nh = pl.hmap.size();
  // (any failure below releases what was created: no leaked context, stream or device memory)
  cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMalloc(&c->d_maps, sizeof(int) * (nj + nh + 36 + 12));
  if (e == cudaSuccess) e = cudaMemcpy(c->d_maps, pl.jmap.data(), sizeof(int) * nj, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(c->d_maps + nj, pl.hmap.data(), sizeof(int) * nh, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(c->d_maps + nj + nh, pl.jbnd, sizeof(int) * 36, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(c->d_maps + nj + nh + 36, pl.hterm, sizeof(int) * 12, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    landing_destroy(c);
    return fail(LANDING_ERR_CUDA, std::string("landing_create: ") + cudaGetErrorString(e));
  }
  c->dpl = DevicePlan{pl.N, pl.nx, pl.np, pl.m, pl.nnzJ, pl.nnzH, pl.off,
                      c->d_maps, c->d_maps + nj, c->d_maps + nj + nh, c->d_maps + nj + nh + 36};
  *out = c;
  return LANDING_OK;
}

void landing_destroy(landing_ctx* c) {
  if (!c) return;
  DeviceGuard guard_(c->device);
  const cudaStream_t st = c->stream;
  solver_free(c->ws);
  if (c->d_maps) cudaFree(c->d_maps);
  if (c->d_kino) cudaFree(c->d_kino);
  if (c->d_khess) cudaFree(c->d_khess);
  if (c->d_kstep) cudaFree(c->d_kstep);
  delete c;  // (the grow-only buffers)
  if (st) cudaStreamDestroy(st);
}

int landing_dims(const landing_ctx* c, long long d[6]) {
  if (!c) return fail(LANDING_ERR_ARG, "landing_dims: null ctx");
  return landing_dims_for(c->N, d);
}

const long long* landing_sparsity(const landing_ctx* c, int which) {
  return c ? landing_sparsity_for(c->N, which) : nullptr;
}

long long landing_launch_count(const landing_ctx* c) { return c ? c->launches : 0; }

int landing_synchronize(landing_ctx* c) {
  if (!c) return fail(LANDING_ERR_ARG, "landing_synchronize: null ctx");
  DeviceGuard guard_(c->device);
  CU(cudaStreamSynchronize(c->stream));
  return LANDING_OK;
}

// ---------------------------------------------------------------- kino-dynamic NLP (SURVEY 8 f-2)
static std::shared_ptr<const KinoPlan> get_kino_plan(int N) {
  static std::mutex mu;
  static std::map<int, std::shared_ptr<const KinoPlan>> cache;
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(N);
  if (it != cache.end()) return it->second;
  auto pl = std::make_shared<const KinoPlan>(make_kino_plan(N));
  cache[N] = pl;
  return pl;
}

int landing_kino_dims(int N, long long d[4]) {
  if (N < 3 || !d) return fail(LANDING_ERR_ARG, "landing_kino_dims: need N >= 3");
  auto pl = get_kino_plan(N);
  d[0] = N; d[1] = pl->nx; d[2] = pl->m; d[3] = pl->nnz;
  return LANDING_OK;
}

const long long* landing_kino_sparsity(int N) { return N < 3 ? nullptr : get_kino_plan(N)->sparsity.data(); }

void landing_kino_setup_default(landing_kino_setup* k) {
  // generate_landingCtrller_KNITRO.m:214-262,325; get_robot_model.m:237-241
  std::memset(k, 0, sizeof(*k));
  const double qtmin[6] = {-10, -10, 0.15, -0.1, -0.1, -10}, qtmax[6] = {10, 10, 5, 0.1, 0.1, 10};
  const double qdtmin[6] = {-10, -10, -10, -.5, -.5, -.5}, qdtmax[6] = {10, 10, 10, .5, .5, .5};
  const double QN[12] = {0, 0, 100, 10, 10, 0, 10, 10, 10, 10, 10, 10};
  const double PI = 3.14159265358979323846;
  for (int i = 0; i < 6; i++) {
    k->q_term_min[i] = qtmin[i]; k->q_term_max[i] = qtmax[i];
    k->qd_term_min[i] = qdtmin[i]; k->qd_term_max[i] = qdtmax[i];
  }
  for (int i = 0; i < 12; i++) k->QN[i] = QN[i];
  k->q_term_ref[2] = 0.25;
  k->z_min = 0.075;
  k->l_leg_max = 0.4;
  for (int l = 0; l < 4; l++) {
    k->jpos_min[3 * l] = -PI / 3; k->jpos_min[3 * l + 1] = -PI / 2; k->jpos_min[3 * l + 2] = 0.0;
    k->jpos_max[3 * l] = PI / 3; k->jpos_max[3 * l + 1] = PI / 2; k->jpos_max[3 * l + 2] = 3 * PI / 4;
  }
  k->tau_max[0] = 18.0; k->tau_max[1] = 18.0; k->tau_max[2] = 27.99;
  k->jpos_guess[0] = 0.0; k->jpos_guess[1] = -PI / 4; k->jpos_guess[2] = PI / 2;
}

int landing_kino_setup_batch(landing_ctx* c, long long B, int memspace, int layout, const landing_kino_setup* ks,
                             const double* drops, const double* x_srb, double* lbg, double* ubg, double* x0) {
  if (!c || !ks || !drops || B < 0) return fail(LANDING_ERR_ARG, "landing_kino_setup_batch: bad arguments");
  if (B == 0 || (!lbg && !ubg && !x0)) return LANDING_OK;
  DeviceGuard guard_(c->device);
  auto pl = get_kino_plan(c->N);
  const long long nsrb = 36LL * c->N - 24;
  Piece pc[5] = {input(drops, 12 * B), input(x_srb, nsrb * B), output(lbg, pl->m * B), output(ubg, pl->m * B),
                 output(x0, pl->nx * B)};
  int rc = stage_in(c, memspace, pc, 5);
  if (rc) return rc;
  KinoSetupArgs a{};
  a.N = c->N; a.B = B; a.ks = *ks;
  a.drops = make_cview(pc[0].at<const double>(), 12, B, layout);
  a.x_srb = make_cview(pc[1].at<const double>(), nsrb, B, layout);
  a.lbg = make_view(pc[2].at<double>(), pl->m, B, layout);
  a.ubg = make_view(pc[3].at<double>(), pl->m, B, layout);
  a.x0 = make_view(pc[4].at<double>(), pl->nx, B, layout);
  c->launches += launch_kino_setup(a, c->stream);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 5);
}

int landing_kino_cost_batch(landing_ctx* c, long long B, int memspace, int layout, const landing_kino_setup* ks,
                            const double* x, double* f, double* grad_f) {
  if (!c || !ks || !x || B < 0) return fail(LANDING_ERR_ARG, "landing_kino_cost_batch: bad arguments");
  if (B == 0 || (!f && !grad_f)) return LANDING_OK;
  DeviceGuard guard_(c->device);
  auto pl = get_kino_plan(c->N);
  Piece pc[3] = {input(x, pl->nx * B), output(f, B), output(grad_f, pl->nx * B)};
  int rc = stage_in(c, memspace, pc, 3);
  if (rc) return rc;
  KinoSetupArgs a{};
  a.N = c->N; a.B = B; a.ks = *ks;
  a.x = make_cview(pc[0].at<const double>(), pl->nx, B, layout);
  a.f = make_view(pc[1].at<double>(), 1, B, layout);
  a.grad_f = make_view(pc[2].at<double>(), pl->nx, B, layout);
  c->launches += launch_kino_cost(a, c->stream);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 3);
}

int landing_kino_eval_batch(landing_ctx* c, long long B, int memspace, int layout, const landing_kino_problem* pb,
                            const double* x, double* g, double* jac) {
  if (!c || !pb || !pb->dt || !x || B < 0) return fail(LANDING_ERR_ARG, "landing_kino_eval_batch: bad arguments");
  if (B == 0 || (!g && !jac)) return LANDING_OK;
  DeviceGuard guard_(c->device);
  if (!c->kino) {
    auto pl = get_kino_plan(c->N);
    const size_t n = pl->gpos.size() + pl->bpos.size();
    CU(cudaMalloc(&c->d_kino, sizeof(int) * n));
    CU(cudaMemcpy(c->d_kino, pl->gpos.data(), sizeof(int) * pl->gpos.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_kino + pl->gpos.size(), pl->bpos.data(), sizeof(int) * pl->bpos.size(), cudaMemcpyHostToDevice));
    c->kino = pl;
  }
  const KinoPlan& pl = *c->kino;
  int rc = stage_dt(c, pb->dt, 0.0);
  if (rc) return rc;
  // AoS batches (one vector per scenario, what landing_solve_batch / landing_kino_setup_batch hand over) are evaluated
  // on transposed copies like the SRB functions (landing_eval_batch)
  Piece pc[3] = {input(x, pl.nx * B), output(g, pl.m * B), output(jac, pl.nnz * B)};
  rc = stage_in(c, memspace, pc, 3);
  if (!rc) rc = aos_to_soa(c, B, &layout, pc, 3);
  if (rc) return rc;
  KinoArgs a{};
  a.N = c->N; a.B = B;
  a.x = make_cview(pc[0].at<const double>(), pl.nx, B, layout);
  a.g = make_view(pc[1].at<double>(), pl.m, B, layout);
  a.jac = make_view(pc[2].at<double>(), pl.nnz, B, layout);
  a.pr.mu = pb->mu; a.pr.mass = pb->mass;
  for (int i = 0; i < 3; i++) { a.pr.Ib[i] = pb->Ib[i]; a.pr.Ib_inv[i] = pb->Ib_inv[i]; }
  a.dtv = c->d_dt.as<double>();
  a.gpos = c->d_kino; a.bpos = c->d_kino + pl.gpos.size();
  c->launches += launch_kino(a, g != nullptr, jac != nullptr, c->stream);
  CU(cudaGetLastError());
  soa_to_aos(c, B, pc, 3);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 3);
}

static std::shared_ptr<const KinoHessPlan> get_kino_hess_plan(int N) {
  static std::mutex mu;
  static std::map<int, std::shared_ptr<const KinoHessPlan>> cache;
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(N);
  if (it != cache.end()) return it->second;
  auto pl = std::make_shared<const KinoHessPlan>(make_kino_hess_plan(N));
  cache[N] = pl;
  return pl;
}

const long long* landing_kino_hess_sparsity(int N) {
  if (N < 3) return nullptr;
  auto pl = get_kino_hess_plan(N);
  if (!pl->err.empty()) {
    g_err = pl->err;
    return nullptr;
  }
  return pl->sparsity.data();
}

int landing_kino_hess_batch(landing_ctx* c, long long B, int memspace, int layout, const landing_kino_problem* pb,
                            const landing_kino_setup* ks, const double* x, const double* lam_f, const double* lam_g,
                            double* hess) {
  if (!c || !pb || !pb->dt || !x || !hess || B < 0 || (lam_f && !ks))
    return fail(LANDING_ERR_ARG, "landing_kino_hess_batch: bad arguments (lam_f needs ks)");
  if (B == 0) return LANDING_OK;
  DeviceGuard guard_(c->device);
  if (!c->khess) {
    auto pl = get_kino_hess_plan(c->N);
    if (!pl->err.empty()) return fail(LANDING_ERR_ARG, pl->err);
    const size_t n = pl->hpos.size() + pl->cpos.size() + pl->rows.size();
    CU(cudaMalloc(&c->d_khess, sizeof(int) * n));
    CU(cudaMemcpy(c->d_khess, pl->hpos.data(), sizeof(int) * pl->hpos.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_khess + pl->hpos.size(), pl->cpos.data(), sizeof(int) * 12, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_khess + pl->hpos.size() + 12, pl->rows.data(), sizeof(unsigned) * pl->rows.size(),
                  cudaMemcpyHostToDevice));
    c->khess = pl;
  }
  const KinoHessPlan& pl = *c->khess;
  const long long m = 48 + 141LL * (c->N - 2) + 117;
  int rc = stage_dt(c, pb->dt, 0.0);
  if (rc) return rc;
  // x, lam_g and hess of AoS batches on transposed copies (landing_kino_eval_batch); lam_f is [B] in both layouts
  Piece pc[4] = {input(x, pl.nx * B), input(lam_g, m * B), output(hess, pl.nnz * B), input(lam_f, B)};
  rc = stage_in(c, memspace, pc, 4);
  if (!rc) rc = aos_to_soa(c, B, &layout, pc, 3);
  if (rc) return rc;
  KinoHessArgs a{};
  a.N = c->N; a.B = B;
  a.x = make_cview(pc[0].at<const double>(), pl.nx, B, layout);
  a.lam_g = make_cview(pc[1].at<const double>(), m, B, layout);
  a.hess = make_view(pc[2].at<double>(), pl.nnz, B, layout);
  a.lam_f = make_cview(pc[3].at<const double>(), 1, B, layout);
  a.pr.mu = pb->mu; a.pr.mass = pb->mass;
  for (int i = 0; i < 3; i++) { a.pr.Ib[i] = pb->Ib[i]; a.pr.Ib_inv[i] = pb->Ib_inv[i]; }
  for (int i = 0; i < 12; i++) a.QN[i] = lam_f ? ks->QN[i] : 0.0;
  a.dtv = c->d_dt.as<double>();
  a.hpos = c->d_khess;
  a.cpos = c->d_khess + pl.hpos.size();
  a.rows = reinterpret_cast<const unsigned*>(c->d_khess + pl.hpos.size() + 12);
  c->launches += launch_kino_hess(a, c->stream);
  CU(cudaGetLastError());
  soa_to_aos(c, B, pc, 3);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 4);
}

// Launches of one call (B > 0, at least one output):
//   6 gradient kernels            if grad_x or dual_inf is wanted
// + 1 g kernel (k_kino_g)         if viol or compl_inf is wanted
// + 1 residual kernel             if viol, dual_inf or compl_inf is wanted
// + for AoS batches of B >= 64: 1 transpose of x, 1 of lam_g if given, 2 of lbg / ubg if given, 1 of grad_x if wanted.
// For example grad_x alone: 6 (SoA) or 8 (AoS, B >= 64, lam_g given); all four outputs with lam_g and the bounds: 8 (SoA)
// or 13 (AoS, B >= 64).
int landing_kino_kkt_batch(landing_ctx* c, long long B, int memspace, int layout, const landing_kino_problem* pb,
                           const landing_kino_setup* ks, const landing_kino_kkt_io* io) {
  if (!c || !pb || !pb->dt || !io || !io->x || B < 0)
    return fail(LANDING_ERR_ARG, "landing_kino_kkt_batch: bad arguments");
  if (io->lam_f && !ks) return fail(LANDING_ERR_ARG, "landing_kino_kkt_batch: lam_f needs ks");
  if (!io->lbg != !io->ubg) return fail(LANDING_ERR_ARG, "landing_kino_kkt_batch: give both lbg and ubg, or neither");
  if ((io->viol || io->compl_inf) && !io->lbg)
    return fail(LANDING_ERR_ARG, "landing_kino_kkt_batch: viol and compl_inf need lbg / ubg");
  const bool want_grad = io->grad_x || io->dual_inf, want_g = io->viol || io->compl_inf;
  const bool want_res = want_g || io->dual_inf;
  if (B == 0 || (!want_grad && !want_res)) return LANDING_OK;
  DeviceGuard guard_(c->device);
  auto pl = get_kino_plan(c->N);
  const long long nx = pl->nx, m = pl->m;
  int rc = stage_dt(c, pb->dt, 0.0);
  if (rc) return rc;
  // x, lam_g, the bounds and grad_x of AoS batches on transposed copies (landing_kino_eval_batch); the others are [B]
  Piece pc[9] = {input(io->x, nx * B),     input(io->lam_g, m * B), input(io->lbg, m * B), input(io->ubg, m * B),
                 output(io->grad_x, nx * B), input(io->lam_f, B),   output(io->viol, B),   output(io->dual_inf, B),
                 output(io->compl_inf, B)};
  rc = stage_in(c, memspace, pc, 9);
  if (!rc) rc = aos_to_soa(c, B, &layout, pc, 5);
  if (rc) return rc;
  // scratch (SoA): g [m x B], and grad_x [n_x x B] when only its norm is wanted
  const bool own_grad = io->dual_inf && !io->grad_x;
  CU(c->kkt.reserve(sizeof(double) * ((want_g ? m : 0) + (own_grad ? nx : 0)) * B));
  double* const g_s = want_g ? c->kkt.as<double>() : nullptr;
  double* const gx_s = own_grad ? c->kkt.as<double>() + (want_g ? m * B : 0) : nullptr;
  const CView x = make_cview(pc[0].at<const double>(), nx, B, layout);
  const View grad = own_grad ? make_view(gx_s, nx, B, LANDING_SOA) : make_view(pc[4].at<double>(), nx, B, layout);
  kino::Params pr{pb->mu, pb->mass, {pb->Ib[0], pb->Ib[1], pb->Ib[2]}, {pb->Ib_inv[0], pb->Ib_inv[1], pb->Ib_inv[2]}};
  if (want_grad) {
    KinoGradArgs a{};
    a.N = c->N; a.B = B;
    a.x = x;
    a.lam_f = make_cview(pc[5].at<const double>(), 1, B, layout);
    a.lam_g = make_cview(pc[1].at<const double>(), m, B, layout);
    a.grad = grad;
    a.pr = pr;
    for (int i = 0; i < 12; i++) {
      a.QN[i] = io->lam_f ? ks->QN[i] : 0.0;
      a.ref[i] = !io->lam_f ? 0.0 : i < 6 ? ks->q_term_ref[i] : ks->qd_term_ref[i - 6];
    }
    a.dtv = c->d_dt.as<double>();
    c->launches += launch_kino_grad(a, c->stream);
  }
  if (want_g) {
    KinoArgs a{};
    a.N = c->N; a.B = B;
    a.x = x;
    a.g = make_view(g_s, m, B, LANDING_SOA);
    a.pr = pr;
    a.dtv = c->d_dt.as<double>();
    c->launches += launch_kino(a, true, false, c->stream);
  }
  if (want_res) {
    KinoKktArgs a{};
    a.B = B; a.m = m; a.nx = nx;
    a.x = x;
    a.lam_f = make_cview(pc[5].at<const double>(), 1, B, layout);
    a.lam_g = make_cview(pc[1].at<const double>(), m, B, layout);
    a.lbg = make_cview(pc[2].at<const double>(), m, B, layout);
    a.ubg = make_cview(pc[3].at<const double>(), m, B, layout);
    a.g = make_view(g_s, m, B, LANDING_SOA);
    a.grad = io->dual_inf ? grad : View{nullptr, 0, 0};
    a.viol = make_view(pc[6].at<double>(), 1, B, layout);
    a.dual_inf = make_view(pc[7].at<double>(), 1, B, layout);
    a.compl_inf = make_view(pc[8].at<double>(), 1, B, layout);
    c->launches += launch_kino_kkt(a, c->stream);
  }
  CU(cudaGetLastError());
  soa_to_aos(c, B, pc, 5);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 9);
}

// Launches of one call (B > 0): 1 step kernel (k_kino_step), + for AoS batches of B >= 64 the transposes of the ten
// [B x n] inputs and of the five [B x n] outputs: 1 (SoA, or AoS with B < 64) or 16 (AoS, B >= 64).
int landing_kino_step_batch(landing_ctx* c, long long B, int memspace, int layout, const landing_kino_step_io* io) {
  if (!c || !io || B < 0) return fail(LANDING_ERR_ARG, "landing_kino_step_batch: bad arguments");
  const void* req[] = {io->g, io->jac, io->hess, io->grad_f, io->s, io->y, io->zL, io->zU, io->lbg, io->ubg, io->mu,
                       io->dw_last, io->dx, io->ds, io->dy, io->dzL, io->dzU, io->delta_w, io->n_factor, io->status};
  for (const void* p : req)
    if (!p) return fail(LANDING_ERR_ARG, "landing_kino_step_batch: a required pointer is NULL");
  if (!io->alpha_pr != !io->alpha_du)
    return fail(LANDING_ERR_ARG, "landing_kino_step_batch: give both alpha_pr and alpha_du, or neither");
  if (io->alpha_pr && !(io->tau > 0.0 && io->tau < 1.0))
    return fail(LANDING_ERR_ARG, "landing_kino_step_batch: tau must be in (0, 1) with the alpha outputs");
  if (B == 0) return LANDING_OK;
  DeviceGuard guard_(c->device);
  if (!c->kstep) {
    auto hp = get_kino_hess_plan(c->N);
    if (!hp->err.empty()) return fail(LANDING_ERR_ARG, hp->err);
    auto pl = std::make_shared<KinoStepHost>();
    const std::string err = make_kino_step_tables(c->N, get_kino_plan(c->N)->sparsity.data(), hp->sparsity.data(), pl.get());
    if (!err.empty()) return fail(LANDING_ERR_ARG, err);
    CU(cudaMalloc(&c->d_kstep, sizeof(int) * (pl->flat.size() + 1)));
    CU(cudaMemcpy(c->d_kstep, pl->flat.data(), sizeof(int) * pl->flat.size(), cudaMemcpyHostToDevice));
    cudaError_t e = cudaSuccess;
    c->kstep_grid = kino_step_resident(&e);
    CU(e);
    c->kstep = pl;
  }
  const KinoStepHost& pl = *c->kstep;
  const long long nx = pl.nx, m = pl.m, nnzJ = get_kino_plan(c->N)->nnz, nnzH = get_kino_hess_plan(c->N)->nnz;
  // the [B x n] arrays of AoS batches on transposed copies (landing_kino_eval_batch); the others are [B]
  Piece pc[22] = {input(io->g, m * B),    input(io->jac, nnzJ * B), input(io->hess, nnzH * B), input(io->grad_f, nx * B),
                  input(io->s, m * B),    input(io->y, m * B),      input(io->zL, m * B),      input(io->zU, m * B),
                  input(io->lbg, m * B),  input(io->ubg, m * B),    output(io->dx, nx * B),    output(io->ds, m * B),
                  output(io->dy, m * B),  output(io->dzL, m * B),   output(io->dzU, m * B),    input(io->mu, B),
                  input(io->dw_last, B),  output(io->delta_w, B),   output(io->n_factor, B),   output(io->status, B),
                  output(io->alpha_pr, B), output(io->alpha_du, B)};
  int rc = stage_in(c, memspace, pc, 22);
  if (!rc) rc = aos_to_soa(c, B, &layout, pc, 15);
  if (rc) return rc;
  const int grid = (int)std::min<long long>(B, c->kstep_grid);
  const long long slot = kino_step_slot(c->N);
  CU(c->kstep_scr.reserve(sizeof(double) * slot * grid));
  KinoStepArgs a{};
  a.B = B;
  a.tb = kino_step_view(pl, c->d_kstep);
  const long long n[15] = {m, nnzJ, nnzH, nx, m, m, m, m, m, m, nx, m, m, m, m};
  CView* in[10] = {&a.g, &a.jac, &a.hess, &a.grad_f, &a.s, &a.y, &a.zL, &a.zU, &a.lbg, &a.ubg};
  View* out[5] = {&a.dx, &a.ds, &a.dy, &a.dzL, &a.dzU};
  for (int i = 0; i < 10; i++) *in[i] = make_cview(pc[i].at<const double>(), n[i], B, layout);
  for (int i = 0; i < 5; i++) *out[i] = make_view(pc[10 + i].at<double>(), n[10 + i], B, layout);
  a.mu = make_cview(pc[15].at<const double>(), 1, B, layout);
  a.dw_last = make_cview(pc[16].at<const double>(), 1, B, layout);
  a.delta_w = make_view(pc[17].at<double>(), 1, B, layout);
  a.n_factor = pc[18].at<int>();
  a.status = pc[19].at<int>();
  a.alpha_pr = make_view(pc[20].at<double>(), 1, B, layout);
  a.alpha_du = make_view(pc[21].at<double>(), 1, B, layout);
  a.tau = io->tau;
  a.scratch = c->kstep_scr.as<double>();
  a.slot = slot;
  a.counter = c->d_kstep + pl.flat.size();
  CU(cudaMemsetAsync(a.counter, 0, sizeof(int), c->stream));
  c->launches += launch_kino_step(a, grid, c->stream);
  CU(cudaGetLastError());
  soa_to_aos(c, B, pc, 15);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 22);
}

int landing_fp64_peak(landing_ctx* c, double* tflops) {
  if (!c || !tflops) return fail(LANDING_ERR_ARG, "landing_fp64_peak: null argument");
  DeviceGuard guard_(c->device);
  std::string err;
  const int rc = fp64_peak_run(c->stream, tflops, &err);
  if (rc != LANDING_OK) return fail(rc, err);
  c->launches += 4;
  return LANDING_OK;
}
void* landing_stream(const landing_ctx* c) { return c ? (void*)c->stream : nullptr; }

void landing_problem_default(landing_problem* pb) {
  // generate_landingCtrller_IPOPT.m:173-196
  static const double qmin[6] = {-10, -10, 0.1, -10, -10, -10}, qmax[6] = {10, 10, 1.0, 10, 10, 10};
  static const double qdmin[6] = {-10, -10, -10, -40, -40, -40}, qdmax[6] = {10, 10, 10, 40, 40, 40};
  static const double qtmin[6] = {-10, -10, 0.2, -0.1, -0.1, -10}, qtmax[6] = {10, 10, 5, 0.1, 0.1, 10};
  static const double qtref[6] = {0, 0, 0.275, 0, 0, 0};
  static const double QN[12] = {0, 0, 100, 100, 100, 0, 10, 10, 10, 10, 10, 10};
  static const double sgn[12] = {1, -1, 1, 1, 1, 1, -1, -1, 1, -1, 1, 1};
  static const double cr[3] = {0.2, 0.1, -0.2};
  pb->T = 0.6;
  for (int i = 0; i < 6; i++) {
    pb->q_min[i] = qmin[i]; pb->q_max[i] = qmax[i];
    pb->qd_min[i] = qdmin[i]; pb->qd_max[i] = qdmax[i];
    pb->q_term_min[i] = qtmin[i]; pb->q_term_max[i] = qtmax[i];
    pb->qd_term_min[i] = qdmin[i]; pb->qd_term_max[i] = qdmax[i];
    pb->q_term_ref[i] = qtref[i]; pb->qd_term_ref[i] = 0.0;
  }
  for (int i = 0; i < 12; i++) { pb->QN[i] = QN[i]; pb->c_ref[i] = sgn[i] * cr[i % 3]; }
  pb->mu = 1.0;
  pb->l_leg_max = 0.35;
  pb->f_max = 200.0;
  for (int i = 0; i < 3; i++) pb->Qf[i] = 0.0;
  pb->kin_box[0] = 0.15; pb->kin_box[1] = 0.15; pb->kin_box[2] = 0.30;
  pb->dt = nullptr;  // uniform T/(N-1)
  pb->formulation = 0;
  pb->cs = nullptr;
  for (int i = 0; i < 12; i++) pb->QX[i] = 0.0;
  pb->delta_c = 1e-7;
  // composite rigid-body inertia at q_home (get_mass_matrix.m:19-54, generate_landingCtrller_IPOPT.m:99-104)
  pb->mass = 8.251999999999999;
  pb->Ib[0] = 0.05757729852959269; pb->Ib[1] = 0.23400899479539086; pb->Ib[2] = 0.2796738482657981;
  pb->Ib_inv[0] = 17.37746888893693; pb->Ib_inv[1] = 4.27334000932043; pb->Ib_inv[2] = 3.577551923825657;
}

void landing_options_default(landing_options* o) {
  // generate_landingCtrller_IPOPT.m:232-263
  std::memset(o, 0, sizeof(*o));
  o->max_iter = 3000;
  o->tol = 1e-4;
  o->constr_viol_tol = 1e-3;
  o->dual_inf_tol = 1.0;
  o->compl_inf_tol = 1e-4;
  o->mu_init = 0.1;
  o->bound_push = 0.5;
  o->bound_frac = 0.5;
  o->bound_relax_factor = 1e-6;
  o->max_soc = 4;
  o->jam_iters = 5;
  o->max_restarts = 8;
  o->jam_alpha = 0.02;
  o->restart_mu = 0.0;  // = mu_init
}

int landing_eval_batch(landing_ctx* c, long long B, int memspace, int layout, const landing_eval_io* io) {
  if (!c || !io || B < 0) return fail(LANDING_ERR_ARG, "landing_eval_batch: bad arguments");
  if (B == 0) return LANDING_OK;
  DeviceGuard guard_(c->device);
  const DevicePlan& pl = c->dpl;
  const long long nx = pl.nx, np = pl.np, m = pl.m, nj = pl.nnzJ, nh = pl.nnzH;
  Piece pc[12] = {input(io->x, nx * B), input(io->p, np * B), input(io->lam_f, B), input(io->lam_g, m * B),
                  output(io->f, B), output(io->g, m * B), output(io->grad_f, nx * B), output(io->jac, nj * B),
                  output(io->hess, nh * B), output(io->grad_x, nx * B), output(io->grad_p, np * B),
                  output(io->status, B)};
  static const bool no_zc = getenv("LANDING_NO_ZEROCOPY") != nullptr;  // restores the staged copies
  const bool zero_copy = memspace == LANDING_HOST && !no_zc && B < 64 && !io->grad_x && !io->grad_p &&
                         staged_bytes(pc, 12) <= (512u << 10);
  int rc = stage_in(c, memspace, pc, 12, zero_copy);
  if (!rc) rc = aos_to_soa(c, B, &layout, pc, 11);  // (status is [B] in both layouts)
  if (rc) return rc;
  EvalArgs a{};
  a.pl = pl;
  a.B = B;
  a.x = make_cview(pc[0].at<const double>(), nx, B, layout);
  a.p = make_cview(pc[1].at<const double>(), np, B, layout);
  a.lam_f = make_cview(pc[2].at<const double>(), 1, B, layout);
  a.lam_g = make_cview(pc[3].at<const double>(), m, B, layout);
  a.f = make_view(pc[4].at<double>(), 1, B, layout);
  a.g = make_view(pc[5].at<double>(), m, B, layout);
  a.grad_f = make_view(pc[6].at<double>(), nx, B, layout);
  a.jac = make_view(pc[7].at<double>(), nj, B, layout);
  a.hess = make_view(pc[8].at<double>(), nh, B, layout);
  a.grad_x = make_view(pc[9].at<double>(), nx, B, layout);
  a.grad_p = make_view(pc[10].at<double>(), np, B, layout);
  a.status = pc[11].at<int>();
  c->launches += launch_eval(a, c->stream);
  CU(cudaGetLastError());
  soa_to_aos(c, B, pc, 11);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 12, zero_copy);
}

void landing_tvlqr_default(landing_tvlqr* q) {
  // quadruped_SRBM_NLP.m:436-475: F = diag(1 1 1, 5 5 5, 4 4 4, 3 3 3, 0...), Q = diag(.25 x3, 1 x3, .5 x3, 1 x3, 0...),
  // R = 90 I, dt = 0.022; inertia at the zero configuration (generateVariationalDynamics.m:4-7; oracle/crba_constants.py)
  static const double f[12] = {1, 1, 1, 5, 5, 5, 4, 4, 4, 3, 3, 3};
  static const double w[12] = {0.25, 0.25, 0.25, 1, 1, 1, 0.5, 0.5, 0.5, 1, 1, 1};
  for (int i = 0; i < 576; i++) q->Q[i] = q->F[i] = 0.0;
  for (int i = 0; i < 12; i++) { q->F[i * 24 + i] = f[i]; q->Q[i * 24 + i] = w[i]; q->R[i] = 90.0; }
  q->T = 0.6;
  q->dt = 0.022;
  q->n_steps = 28;  // T / dt + 1
  static const double Ib[9] = {8.2057376e-02, 0.0, -5.020000000000024e-05, 0.0, 2.46291e-01, 0.0,
                               -5.020000000000024e-05, 0.0, 2.67475776e-01};
  for (int i = 0; i < 9; i++) q->Ib[i] = Ib[i];
  q->mass = 8.251999999999999;
}

int landing_tvlqr_batch(landing_ctx* c, long long B, int memspace, const landing_tvlqr* par, const double* x_star,
                        double* P_out, double* K_out) {
  if (!c || !par || !x_star || B < 0 || par->n_steps < 1) return fail(LANDING_ERR_ARG, "landing_tvlqr_batch: bad arguments");
  if (B == 0) return LANDING_OK;
  DeviceGuard guard_(c->device);
  const long long nx = c->dpl.nx, ns = par->n_steps;
  Piece pc[3] = {input(x_star, nx * B), output(P_out, 576 * ns * B), output(K_out, 288 * ns * B)};
  int rc = stage_in(c, memspace, pc, 3);
  if (rc) return rc;
  TvlqrArgs a{};
  a.N = c->N; a.nx = nx; a.par = *par;
  a.x_star = pc[0].at<const double>(); a.P_out = pc[1].at<double>(); a.K_out = pc[2].at<double>();
  c->launches += launch_tvlqr(a, B, c->stream);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 3);
}

int landing_bounds_batch(landing_ctx* c, long long B, int memspace, int layout, const double* p,
                         double* lbg, double* ubg) {
  if (!c || !p || !lbg || !ubg || B <= 0) return fail(LANDING_ERR_ARG, "landing_bounds_batch: bad arguments");
  DeviceGuard guard_(c->device);
  const DevicePlan& pl = c->dpl;
  Piece pc[3] = {input(p, pl.np * B), output(lbg, pl.m * B), output(ubg, pl.m * B)};
  int rc = stage_in(c, memspace, pc, 3);
  if (rc) return rc;
  c->launches += launch_bounds(pl, B, make_cview(pc[0].at<const double>(), pl.np, B, layout),
                               make_view(pc[1].at<double>(), pl.m, B, layout), make_view(pc[2].at<double>(), pl.m, B, layout),
                               c->stream);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 3);
}

int landing_build_batch(landing_ctx* c, long long B, int memspace, int layout, const landing_problem* pb,
                        const double* drops, double* p, double* x0) {
  if (!c || !pb || !drops || B <= 0) return fail(LANDING_ERR_ARG, "landing_build_batch: bad arguments");
  DeviceGuard guard_(c->device);
  const DevicePlan& pl = c->dpl;
  Piece pc[3] = {input(drops, 12 * B), output(p, pl.np * B), output(x0, pl.nx * B)};
  int rc = stage_in(c, memspace, pc, 3);
  if (!rc) rc = stage_dt(c, pb->dt, pb->T);
  if (!rc) rc = stage_cs(c, pb);
  if (rc) return rc;
  c->launches += launch_build(pl, B, *pb, c->d_dt.as<double>(), pc[0].at<const double>(),
                              make_view(pc[1].at<double>(), pl.np, B, layout), make_view(pc[2].at<double>(), pl.nx, B, layout),
                              c->stream);
  CU(cudaGetLastError());
  return stage_out(c, memspace, pc, 3);
}

int landing_solve_batch(landing_ctx* c, long long B, int memspace, const landing_problem* pb,
                        const landing_options* opt, const landing_solve_io* io) {
  if (!c || !pb || !io || B < 0) return fail(LANDING_ERR_ARG, "landing_solve_batch: bad arguments");
  if (B == 0) return LANDING_OK;  // an empty sweep is a no-op (the reference's sweep loops simply do not iterate)
  if (!io->drops) return fail(LANDING_ERR_ARG, "landing_solve_batch: drops is NULL");
  DeviceGuard guard_(c->device);
  landing_options o;
  if (opt) o = *opt; else landing_options_default(&o);
  int rc = stage_dt(c, pb->dt, pb->T);
  if (!rc) rc = stage_cs(c, pb);
  if (rc) return rc;
  const long long nx = c->dpl.nx, m = c->dpl.m;
  Piece pc[8] = {input(io->drops, 12 * B), input(io->x0, nx * B), output(io->x_star, nx * B), output(io->f_star, B),
                 output(io->lam_g, m * B), output(io->viol, B), output(io->status, B), output(io->iters, B)};
  rc = stage_in(c, memspace, pc, 8);
  if (rc) return rc;
  const landing_solve_io dio{pc[0].at<const double>(), pc[1].at<const double>(), pc[2].at<double>(), pc[3].at<double>(),
                             pc[4].at<double>(), pc[5].at<double>(), pc[6].at<int>(), pc[7].at<int>()};
  std::string err;
  int launches = 0;
  rc = solver_run(c->ws, c->dpl, B, *pb, c->d_dt.as<double>(), pb->formulation == 1 ? c->d_cs.as<unsigned char>() : nullptr,
                  o, dio, c->stream, &launches, &err);
  c->launches += launches;
  if (rc) return fail(rc, err);
  return stage_out(c, memspace, pc, 8);
}

// ---------------------------------------------------------------- several GPUs, one process
struct landing_multi {
  int N = 0;
  std::vector<landing_ctx*> ctx;
  std::vector<PinnedBuf> sh;  // pinned host staging of each device's shard
};

int landing_multi_create(int N, int n_devices, const int* devices, landing_multi** out) {
  if (!out || !devices || n_devices < 1) return fail(LANDING_ERR_ARG, "landing_multi_create: bad arguments");
  std::unique_ptr<landing_multi> m(new landing_multi());
  m->N = N;
  m->sh = std::vector<PinnedBuf>(n_devices);
  for (int d = 0; d < n_devices; d++) {
    landing_ctx* c = nullptr;
    const int rc = landing_create(N, devices[d], &c);
    if (rc) {
      for (landing_ctx* q : m->ctx) landing_destroy(q);
      return rc;
    }
    m->ctx.push_back(c);
  }
  *out = m.release();
  return LANDING_OK;
}

void landing_multi_destroy(landing_multi* m) {
  if (!m) return;
  for (size_t d = 0; d < m->ctx.size(); d++) {
    DeviceGuard guard_(m->ctx[d]->device);
    m->sh[d].release();
    landing_destroy(m->ctx[d]);
  }
  delete m;
}

int landing_solve_batch_multi(landing_multi* m, long long B, const landing_problem* pb, const landing_options* opt,
                              const landing_solve_io* io) {
  if (!m || !pb || !io || B < 0) return fail(LANDING_ERR_ARG, "landing_solve_batch_multi: bad arguments");
  if (B == 0) return LANDING_OK;
  if (!io->drops || !io->x_star || !io->f_star || !io->status || !io->iters)
    return fail(LANDING_ERR_ARG, "landing_solve_batch_multi: drops, x_star, f_star, status and iters are required");
  const int G = (int)m->ctx.size();
  const long long nx = 36LL * m->N - 24, mr = 104LL * m->N - 92;
  std::vector<int> rcs(G, LANDING_OK);
  std::vector<std::string> errs(G);
  auto work = [&](int d) {
    landing_ctx* c = m->ctx[d];
    const long long Bd = (B - d + G - 1) / G;  // scenarios d, d + G, ...
    if (Bd <= 0) return;
    DeviceGuard guard_(c->device);
    const long long nd = (12 + nx + 2 + (io->lam_g ? mr : 0) + (io->x0 ? nx : 0)) * Bd;  // doubles, then 2 Bd ints
    if (m->sh[d].reserve(sizeof(double) * nd + sizeof(int) * 2 * Bd) != cudaSuccess) {
      rcs[d] = LANDING_ERR_CUDA;
      errs[d] = "landing_solve_batch_multi: pinned host allocation failed";
      return;
    }
    landing_solve_io sio{};
    double* p = m->sh[d].as<double>();
    double* drops = p; p += 12 * Bd;
    sio.x_star = p; p += nx * Bd;
    sio.f_star = p; p += Bd;
    sio.viol = p; p += Bd;
    if (io->lam_g) { sio.lam_g = p; p += mr * Bd; }
    double* x0 = io->x0 ? p : nullptr; p += io->x0 ? nx * Bd : 0;
    sio.status = (int*)p;
    sio.iters = sio.status + Bd;
    for (long long i = 0; i < Bd; i++) {
      const long long b = d + i * G;
      std::memcpy(drops + 12 * i, io->drops + 12 * b, sizeof(double) * 12);
      if (x0) std::memcpy(x0 + nx * i, io->x0 + nx * b, sizeof(double) * nx);
    }
    sio.drops = drops; sio.x0 = x0;
    rcs[d] = landing_solve_batch(c, Bd, LANDING_HOST, pb, opt, &sio);
    if (rcs[d]) { errs[d] = landing_last_error(); return; }
    for (long long i = 0; i < Bd; i++) {  // gather: this device's records into the whole sweep's arrays
      const long long b = d + i * G;
      std::memcpy(io->x_star + nx * b, sio.x_star + nx * i, sizeof(double) * nx);
      io->f_star[b] = sio.f_star[i];
      io->status[b] = sio.status[i];
      io->iters[b] = sio.iters[i];
      if (io->viol) io->viol[b] = sio.viol[i];
      if (io->lam_g) std::memcpy(io->lam_g + mr * b, sio.lam_g + mr * i, sizeof(double) * mr);
    }
  };
  std::vector<std::thread> th;
  for (int d = 1; d < G; d++) th.emplace_back(work, d);
  work(0);
  for (auto& t : th) t.join();
  for (int d = 0; d < G; d++)
    if (rcs[d]) return fail(rcs[d], errs[d]);
  return LANDING_OK;
}

}  // extern "C"
