// Internal declarations of the CUDA engine behind include/safe_mpc_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/safe_mpc_b200.h"
#include "qp_split.cuh"

namespace smpc {

constexpr int NN_OUT = 11;   // viability row value + 10 gradient entries

struct MlpWeights {
  // fp32 weights of the reference architecture 10 -> 256 -> 256 -> 256 -> 1 (safe_set.py:26-43)
  const float *W1, *b1, *W2, *b2, *W3, *b3, *W4, *b4;   // row-major [out][in]
  const float *W2t, *W3t;                               // transposed copies [in][out] for the forward sweep
};

// which (problem, stage) rows the viability network is evaluated on
enum { ROWS_TERMINAL = 0, ROWS_ALL = 1, ROWS_RECEDING = 2, ROWS_FLAT = 3, ROWS_CAND = 4 };   // ROWS_CAND: one row per problem, at stage r[b]

// operands of the tensor-core evaluation of the network (mlp_tc.cu): plain fp32 vectors + the packed hi / lo stage images
struct MlpTcWeights {
  const float *W1, *b1, *b2, *b3, *W4, *b4;
  const float* packed;          // stage images of the single-CTA kernel (mlp_tc.cu)
  const float* packed2;         // stage images per CTA of the pair kernel (mlp_tc2.cu)
};

#if defined(__CUDACC__)
// row i of an evaluation -> (problem b, stage k); false when the row is not evaluated
__device__ __forceinline__ bool mlp_row(int rows_mode, int i, int B, int N, const int32_t* r, const uint8_t* act, const uint8_t* need,
                                        int& b, int& k) {
  if (rows_mode == ROWS_TERMINAL) { b = i; k = N; }
  else if (rows_mode == ROWS_ALL) { b = i / N; k = 1 + i % N; }
  else if (rows_mode == ROWS_RECEDING) { b = i >> 1; if (b >= B) return false; k = (i & 1) ? N : r[b]; if (k < 1 || (!(i & 1) && k >= N)) return false; }
  else if (rows_mode == ROWS_CAND) { b = i; if (b >= B) return false; k = r[b]; if (k < 1 || k > N) return false; }
  else { b = i; k = 0; return true; }
  if (b >= B) return false;
  if (act && !act[b]) return false;
  if (need && !need[b]) return false;
  return true;
}
#endif

struct LaunchCtx {
  cudaStream_t stream;
  int64_t* launches;
};

// kernels.cu
cudaError_t mlp_prepare();
cudaError_t linearize_prepare();
void launch_prep(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, double* xg, const double* ug, const uint8_t* act, bool correct);
void launch_mlp(const LaunchCtx& c, const smpc_problem_t* dP, const MlpWeights& w, int B, int N, int rows_mode, int n_flat,
                const double* xsrc, const int32_t* r, const uint8_t* act, const uint8_t* need, double* out11, bool want_grad);
// mlp_tc.cu -- the same evaluation on the tensor cores (fp32 class, smpc_problem_t::nn_precision = 1)
size_t mlp_tc_packed_floats();
void mlp_tc_pack(const float* W2, const float* W3, float* out);
cudaError_t mlp_tc_prepare();
void launch_mlp_tc(const LaunchCtx& c, const smpc_problem_t* dP, const MlpTcWeights& w, int n_sm, int B, int N, int rows_mode, int n_flat,
                   const double* xsrc, const int32_t* r, const uint8_t* act, const uint8_t* need, double* out11, bool want_grad);
// mlp_tc2.cu -- CTA-pair form (tcgen05 cta_group::2, thread-block cluster of two)
size_t mlp_tc2_packed_floats();
void mlp_tc2_pack(const float* W2, const float* W3, float* out);
cudaError_t mlp_tc2_prepare();
void launch_mlp_tc2(const LaunchCtx& c, const smpc_problem_t* dP, const MlpTcWeights& w, int n_sm, int B, int N, int rows_mode, int n_flat,
                    const double* xsrc, const int32_t* r, const uint8_t* act, const uint8_t* need, double* out11, bool want_grad);
// lin: tile-interleaved record array of the QP solver, double or (lin_f32) float
void launch_linearize(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, const double* xg, const double* ug,
                      const int32_t* r, const uint8_t* act, const double* nn11, const double* traj, int n_traj, const int32_t* cur_step,
                      void* lin, bool lin_f32);
void launch_ctrl_post1(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, const uint8_t* act, const double* xg, const double* ug,
                       const double* xt, int32_t* status, int32_t* fails, int32_t* r, double* x_viable, uint8_t* need_scan,
                       uint8_t* abort_flag, double* u_out);
void launch_ctrl_post2(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, const uint8_t* act, double* xg, double* ug,
                       const double* xt, const double* ut, const int32_t* fails, int32_t* r, int32_t* cur_step,
                       const uint8_t* need_scan, const double* scan11, const uint8_t* abort_flag, double* u_out);
// ParallelController (controller.py:567-644): bookkeeping of the candidate-node loop
void launch_par_begin(const LaunchCtx& c, int B, const uint8_t* act, int32_t* best, uint8_t* done, uint8_t* act2, int* n_open);
void launch_par_eval(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, int n, const uint8_t* act2_in, const int32_t* status, const int32_t* r,
                     const double* xt, const double* ut, const double* scan11, int32_t* best, double* best_xt, double* best_ut, uint8_t* done,
                     uint8_t* act2_out, int* n_open);
void launch_par_post(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, const uint8_t* act, const double* xg, const double* ug, double* xt,
                     double* ut, const int32_t* best, const double* best_xt, const double* best_ut, int32_t* fails, int32_t* r, double* x_viable,
                     uint8_t* need_scan, uint8_t* abort_flag, double* u_out);
void launch_plant(const LaunchCtx& c, const smpc_problem_t* dP, int B, const double* inertial, const double* noise, const double* x,
                  const double* u, const uint8_t* act, double* xn, double* a);
void launch_tau(const LaunchCtx& c, const smpc_problem_t* dP, int n, const double* x, const double* u, double* tau);
void launch_rk4_sens(const LaunchCtx& c, const smpc_problem_t* dP, int n, double dt, const double* x, const double* tau, double* xn, double* A, double* B);
void launch_kin(const LaunchCtx& c, const smpc_problem_t* dP, int n, const double* x, double* ee, double* dist);
void launch_fill_i32(const LaunchCtx& c, int32_t* p, int n, int32_t v);
void launch_fill_f64(const LaunchCtx& c, double* p, size_t n, double v);
void launch_set_xviable_from_guess(const LaunchCtx& c, int B, int N, const double* xg, double* xv);

// sim kernels
struct SimDev {
  int B, N, Nb, n_steps;
  double *x, *xlog, *ulog, *x_abort, *u_abort, *xv_first, *u_ctrl, *u;
  int32_t *mode, *ja, *outcome;
  uint8_t *need_ctrl, *need_backup, *abort_flag, *live;
  unsigned long long* counters;   // [SIM_NCOUNTERS]: RTI solves, backup solves, plant steps, IPM iterations; [4] = backup requests so far (host: skip the
                                  // empty backup solve); then the device-side step bookkeeping of captured steps (below)
};
enum { SIM_REQ_SEEN = 5,          // backup requests at the start of the current captured step
       SIM_STEP_CUR = 6,          // index of the current captured step
       SIM_STEP_NEXT = 7,         // index of the next step (written by every step, eager or captured)
       SIM_NCOUNTERS = 8 };
void launch_sim_pre(const LaunchCtx& c, const SimDev& s, const smpc_problem_t* dP, int j);
void launch_sim_mid(const LaunchCtx& c, const SimDev& s, const double* x_viable, double* bk_xg, double* bk_ug, const int32_t* qp_iter_main);
void launch_sim_post(const LaunchCtx& c, const SimDev& s, const smpc_problem_t* dP, int j, const int32_t* bk_status, const double* bk_xt,
                     const double* bk_ut, const double* inertial, const double* noise, const int32_t* qp_iter_bk);
void launch_sim_outcome(const LaunchCtx& c, const SimDev& s, const smpc_problem_t* dP, int32_t* out);
void launch_sim_backup_cond(const LaunchCtx& c, const SimDev& s, cudaGraphConditionalHandle cond);

// qp.cu -- split interior-point solver (qp_split.cuh).  The library holds it twice: qp.cu (fp64 storage, namespace smpc::f64) and
// qp_f32.cu (the same source with QS_REAL = float, namespace smpc::f32); the flavour of this translation unit is an inline namespace.
#define SMPC_QP_API                                                                                                                       \
  struct QpSolver;                                                                                                                        \
  size_t qp_bytes(int B, int N);                                                                                                          \
  QpSolver* qp_create(int B, int N, int iter_max, bool keep_slots, cudaStream_t stream, cudaError_t* err);                                \
  void qp_destroy(QpSolver* s);                                                                                                           \
  void* qp_rec(QpSolver* s);               /* tile-interleaved stage records [T][N+1][REC][32] the linearisation writes (storage type) */ \
  int qp_groups(const QpSolver* s);        /* tile groups solved concurrently */                                                          \
  int qp_last_iterations(const QpSolver* s);                                                                                              \
  int qp_compactions(const QpSolver* s);   /* compactions of the slots during the last solve (> 0: per-slot dumps are gone) */            \
  void qp_set_profiling(QpSolver* s, bool on);                                                                                            \
  bool qp_traced(const QpSolver* s);       /* profiling or SMPC_QP_TRACE: the solve reads events back on the host */                      \
  void qp_get_profile(const QpSolver* s, double* ms, int32_t* n, double* span_ms);                                                        \
  /* one batched solve; reads the records of qp_rec(); problems with act == 0 are skipped and keep their outputs */                      \
  cudaError_t launch_qp_solve(const LaunchCtx& c, const smpc_problem_t* dP, QpSolver* s, const double* x0, const int32_t* r,              \
                              const uint8_t* act, double* xt, double* ut, int32_t* status, int32_t* qp_iter, int32_t* qp_status,          \
                              double* qp_res);                                                                                            \
  void launch_rec_untile(const LaunchCtx& c, QpSolver* s, double* out);                                                                   \
  void launch_dump_qp(const LaunchCtx& c, const smpc_problem_t* dP, QpSolver* s, double* dz, double* pi, double* lam, double* t);
inline namespace QS_FLAVOUR {
SMPC_QP_API
}  // inline namespace QS_FLAVOUR
namespace QS_OTHER_FLAVOUR {
SMPC_QP_API
}

}  // namespace smpc
