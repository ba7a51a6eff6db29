// kino_step.cu -- batched primal-dual Newton step of the kino-dynamic ("full-body") landing NLP (include/landing_b200.h:
// landing_kino_step_batch), with IPOPT's inertia correction.  One CTA per scenario on a persistent grid: the CTAs pull
// scenario ids from a counter, so the factor scratch (STEP_STAGE doubles per stage) grows with the resident CTAs, not with
// B.  Per scenario: the interior test, then the backward Riccati sweep over the N-1 stages with the 60 x 60 stage matrix
// in shared memory, repeated with a larger dw while a control block has a pivot <= 1e-14, then the forward sweep and the
// recovery of ds, dy, dzL, dzU (parallel over rows) with the fraction-to-boundary step lengths.  The maths, shared with
// the host build, is in kino_step.cuh.
#include "kernels.cuh"
#include "kino_step.cuh"

namespace srb {
namespace {

constexpr int STEP_NT = 256;

struct DevIn {
  CView jac_, hess_, gf_;
  long long b;
  __device__ __forceinline__ double jac(long long i) const { return jac_.get(i, b); }
  __device__ __forceinline__ double hess(long long i) const { return hess_.get(i, b); }
  __device__ __forceinline__ double gf(long long i) const { return gf_.get(i, b); }
};
__device__ __forceinline__ kino::SV sv(const CView& v, long long b) { return {v.p + b * v.sb, v.si}; }
__device__ __forceinline__ kino::MV mv(const View& v, long long b) { return {v.p + b * v.sb, v.si}; }

__global__ void __launch_bounds__(STEP_NT) k_kino_step(KinoStepArgs a) {
  extern __shared__ double smem[];
  __shared__ long long s_b;
  __shared__ double s_red[2][STEP_NT / 32];
  kino::StepShared sh(smem);
  const kino::Team tm{(int)threadIdx.x, STEP_NT};
  double* scr = a.scratch + (size_t)blockIdx.x * a.slot;
  const double QNAN = __longlong_as_double(0x7ff8000000000000LL);
  for (;;) {
    if (threadIdx.x == 0) s_b = atomicAdd(a.counter, 1);
    __syncthreads();
    const long long b = s_b;
    __syncthreads();
    if (b >= a.B) return;
    const DevIn in{a.jac, a.hess, a.grad_f, b};
    const kino::StepPoint it{sv(a.g, b), sv(a.s, b), sv(a.y, b), sv(a.zL, b), sv(a.zU, b), sv(a.lbg, b), sv(a.ubg, b),
                             a.mu.get(0, b)};
    const kino::StepOut o{mv(a.dx, b), mv(a.ds, b), mv(a.dy, b), mv(a.dzL, b), mv(a.dzU, b)};
    const double dw_last = a.dw_last.get(0, b);
    int status = 0, nf = 0;
    double dw = QNAN;
    if (__syncthreads_and(kino::step_interior(it, a.tb.m, tm))) {
      dw = kino::dw_first(dw_last);
      for (int tries = 0;;) {
        nf++;
        if (kino::step_factor(a.tb, in, it, dw, sh, scr, tm)) break;
        dw = kino::dw_next(dw, dw_last, tries);
        tries++;
        if (dw > 1e40) { status = LANDING_ST_FACTOR_FAIL; break; }
      }
    } else {
      status = LANDING_ST_NOT_INTERIOR;
    }
    double apr = QNAN, adu = QNAN;
    if (status == 0) {
      kino::step_solve(a.tb, in, it, scr, sh, o, a.tau, &apr, &adu, tm);
      if (a.alpha_pr.p) {  // block minima (exact in any order)
        for (int off = 16; off > 0; off >>= 1) {
          apr = fmin(apr, __shfl_xor_sync(0xffffffffu, apr, off));
          adu = fmin(adu, __shfl_xor_sync(0xffffffffu, adu, off));
        }
        if ((threadIdx.x & 31) == 0) { s_red[0][threadIdx.x / 32] = apr; s_red[1][threadIdx.x / 32] = adu; }
        __syncthreads();
        apr = 1.0; adu = 1.0;
        for (int w = 0; w < STEP_NT / 32; w++) { apr = fmin(apr, s_red[0][w]); adu = fmin(adu, s_red[1][w]); }
      }
    } else {  // no step: every output of the scenario is NaN
      for (long long j = threadIdx.x; j < a.tb.nx; j += STEP_NT) o.dx[j] = QNAN;
      for (long long i = threadIdx.x; i < a.tb.m; i += STEP_NT) {
        o.ds[i] = QNAN; o.dy[i] = QNAN; o.dzL[i] = QNAN; o.dzU[i] = QNAN;
      }
    }
    if (threadIdx.x == 0) {
      a.delta_w.at(0, b) = dw;
      a.n_factor[b] = nf;
      a.status[b] = status;
      if (a.alpha_pr.p) { a.alpha_pr.at(0, b) = apr; a.alpha_du.at(0, b) = adu; }
    }
    __syncthreads();  // (s_red and s_b are reused by the next scenario)
  }
}

}  // namespace

// ---------------------------------------------------------------- host
std::string make_kino_step_tables(int N, const long long* jsp, const long long* hsp, KinoStepHost* out) {
  const long long nx = jsp[1];
  const kino::KinoStepPlan pl = kino::make_kino_step_plan(N, jsp + 2, jsp + 2 + nx + 1, hsp + 2, hsp + 2 + nx + 1);
  if (!pl.err.empty()) return pl.err;
  const std::vector<int>* parts[] = {&pl.mstage, &pl.mtgt, &pl.mbeg, &pl.mterm, &pl.qstage, &pl.qtgt,
                                     &pl.qbeg,   &pl.qterm, &pl.dstage, &pl.dterm, &pl.rptr, &pl.rent};
  out->flat.clear();
  for (int i = 0; i < 12; i++) {
    out->off[i] = (long long)out->flat.size();
    out->flat.insert(out->flat.end(), parts[i]->begin(), parts[i]->end());
  }
  out->N = N; out->nx = pl.nx; out->m = pl.m;
  return "";
}

kino::StepTables kino_step_view(const KinoStepHost& h, const int* d) {
  return kino::StepTables{h.N, h.nx, h.m, d + h.off[0], d + h.off[1], d + h.off[2], d + h.off[3], d + h.off[4],
                          d + h.off[5], d + h.off[6], d + h.off[7], d + h.off[8], d + h.off[9], d + h.off[10], d + h.off[11]};
}

int kino_step_smem_bytes() { return kino::STEP_SMEM * (int)sizeof(double); }
long long kino_step_slot(int N) { return (long long)N * kino::STEP_STAGE; }

// resident CTAs of k_kino_step on the current device (the persistent grid; one scratch slot each)
int kino_step_resident(cudaError_t* err) {
  int dev = 0, sms = 0, per = 0;
  *err = cudaGetDevice(&dev);
  if (*err == cudaSuccess) *err = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (*err == cudaSuccess)
    *err = cudaFuncSetAttribute(k_kino_step, cudaFuncAttributeMaxDynamicSharedMemorySize, kino_step_smem_bytes());
  if (*err == cudaSuccess)
    *err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_kino_step, STEP_NT, kino_step_smem_bytes());
  return sms * (per > 0 ? per : 1);
}

int launch_kino_step(const KinoStepArgs& a, int grid, cudaStream_t st) {
  k_kino_step<<<grid, STEP_NT, kino_step_smem_bytes(), st>>>(a);
  return 1;
}

}  // namespace srb
