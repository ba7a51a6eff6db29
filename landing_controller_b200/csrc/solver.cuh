// solver.cuh -- batched primal-dual interior-point solver (declarations)
#pragma once
#include <string>

#include "growbuf.cuh"
#include "kernels.cuh"

namespace srb {

// Host-built, device-resident index tables derived from the knot pattern (interior knot numbering;
// the last knot is remapped onto it).  See solver.cu for the meaning of each table.
struct SolverTables {
  int *dev = nullptr;  // one allocation
  const int *jl_last, *hl_last;            // emission index of the last-knot template -> interior index
  const int *r_ptr, *r_terms;              // per inequality row rho: sum J_e dw[idx]
  const int *c_ptr, *c_terms;              // per local variable (60): sum J_e y_rho  (grad of the Lagrangian)
  // accumulator-tile initialisation of the stage factorisation: for tile (27) x lane (32), the positions of the lane's
  // two entries in the condensed stage data (low / high 16 bits; 0xffff = structurally zero)
  const int *tinit;
  // tables the sweeps keep in SHARED memory (copied once per CTA): offsets into sm_src[0..sm_count)
  const int *sm_src; int sm_count;
  int o_g, n_g;          // dynamics entries: e | (state*36 + var) << 10   -> G
  int o_qptr, o_qterms;  // stage gradient per stage variable (elimination order): (rho << 10) | e, padded to pairs
  // condensing targets of the stage matrix (lower triangle, elimination order m = (s+24) mod 48):
  //   M[a][b] += H[h] (if any) + sum sigma_rho J_ea J_eb over terms (rho<<20 | ea<<10 | eb), padded to pairs
  int o_uabh, o_uptr, o_uterms, n_u;   // uabh = (a*48+b) | (h+1) << 12
  int o_rptr, o_rterms, o_cptr, o_cterms;  // shared-memory copies of the row / column schedules
};

struct SolverWorkspace {
  DeviceBuf scratch;          // per-warp-slot scratch (iterate, lists, Riccati factors)
  int* counter = nullptr;     // work-queue head
  double* zeros = nullptr;    // 16 zeros (c+ operand of the last knot)
  DeviceBuf order;            // work-queue order (scenario ids, longest expected first), and for large sweeps the
                              // sort keys / ids / temporary storage behind it
  unsigned char* kt = nullptr;  // row-kind tables (k_kinds)
  SolverTables tab;
  int n_sm = 0;
  bool ready = false;         // first-call set-up (tables, queue head, kernel attributes) completed
};

// frees the first-call set-up (the grow-only buffers free themselves)
void solver_free(SolverWorkspace& ws);

// FP64 FMA throughput of the device (roofline denominator of the interior-point kernel), TFLOP/s
int fp64_peak_run(cudaStream_t st, double* tflops, std::string* err);

// io: device pointers
int solver_run(SolverWorkspace& ws, const DevicePlan& pl, long long B,
               const landing_problem& pb, const double* dtv, const unsigned char* csm, const landing_options& opt,
               const landing_solve_io& io,
               cudaStream_t st, int* launches, std::string* err);

}  // namespace srb
