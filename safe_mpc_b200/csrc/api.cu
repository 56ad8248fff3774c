// C ABI of the engine (include/safe_mpc_b200.h).  Host-side orchestration only: buffers, streams, kernel sequencing.
// There is no CPU compute path in this library: every entry point that produces numbers launches kernels.
#include <cstdio>
#include <cstring>
#include <vector>

#include "engine.cuh"

using namespace smpc;

namespace {
thread_local std::string g_create_error;

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
};
}  // namespace

struct smpc_handle {
  smpc_problem_t P;
  smpc_problem_t* dP = nullptr;
  int B = 0, N = 0, device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;           // false: the caller's stream (smpc_set_stream), never destroyed here
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  int64_t launches = 0;
  double* ee_traj = nullptr;        // [n_traj][3] end-effector reference per control step (smpc_set_ee_trajectory); n_traj = 0: P.ee_ref
  int n_traj = 0;
  std::string err;
  std::vector<void*> allocs;
  // network
  float* dW = nullptr;
  MlpWeights w{};
  float* dWtc = nullptr;            // packed tf32 hi / lo stage images of the tensor-core path (mlp_tc.cu)
  float* dWtc2 = nullptr;           // the same per CTA of the pair kernel (mlp_tc2.cu)
  bool tc_pair = false;             // SMPC_MLP_TC=pair: the CTA-pair kernel (cta_group::2) instead of one CTA per tile
  MlpTcWeights wtc{};
  int n_sm = 0;
  // state
  double *xg = nullptr, *ug = nullptr, *xt = nullptr, *ut = nullptr, *plant_inertial = nullptr, *tau_noise = nullptr,
         *x_viable = nullptr, *nn11 = nullptr, *scan11 = nullptr, *qp_res = nullptr, *x_in = nullptr, *u_out = nullptr;
  // split interior-point solver: tile-interleaved records + solver state, in the storage flavour the handle was created with
  // (smpc_problem_t::precision): exactly one of the two is set
  f64::QpSolver* qp = nullptr;
  f32::QpSolver* qpf = nullptr;
  const uint8_t* act_last = nullptr;
  bool solved = false;
  int32_t *fails = nullptr, *r = nullptr, *status = nullptr, *qp_iter = nullptr, *qp_status = nullptr, *cur_step = nullptr;
  uint8_t *act = nullptr, *need_scan = nullptr, *abort_flag = nullptr;
  // ParallelController (controller.py:567-644): candidate node of the running solve, best node so far and its trajectory
  int32_t *cand = nullptr, *par_best = nullptr;
  uint8_t *par_done = nullptr, *par_act = nullptr;
  double *par_xt = nullptr, *par_ut = nullptr;
  int* par_open = nullptr;          // device: problems that still have candidates to try
  int* h_par_open = nullptr;        // pinned
  // staging for host callers
  void* stage = nullptr;
  size_t stage_bytes = 0;
  double times[7] = {0, 0, 0, 0, 0, 0, 0};
  bool timed = false;
  int times_pending = 0;        // 1: events of an rti_solve recorded, 2: of a controller_step; collected by smpc_get_times
  LaunchCtx ctx() { return LaunchCtx{stream, &launches}; }
};

struct smpc_sim {
  smpc_handle* c;
  smpc_handle* bk;
  SimDev d;
  int j = 0;
  int32_t* outcome_tmp = nullptr;
  unsigned long long* h_requests = nullptr;   // pinned: backup requests so far (SimDev::counters[4])
  unsigned long long requests_seen = 0;
  cudaStream_t body = nullptr;      // captures the body of the conditional backup solve of a captured step
  std::vector<void*> allocs;        // device buffers of this closed loop (freed by smpc_sim_destroy)
  int device = 0;
};

namespace {

// call a QP-solver function of the handle's storage flavour
#define QPCALL(h, fn, ...) ((h)->qpf ? f32::fn((h)->qpf, ##__VA_ARGS__) : f64::fn((h)->qp, ##__VA_ARGS__))

int fail(smpc_handle* h, int code, const char* what, cudaError_t e = cudaSuccess) {
  char buf[512];
  if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
  else snprintf(buf, sizeof buf, "%s", what);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

#define CK(h, call)                                                         \
  do {                                                                      \
    cudaError_t e__ = (call);                                               \
    if (e__ != cudaSuccess) return fail(h, SMPC_ERR_CUDA, #call, e__);      \
  } while (0)

template <class T>
cudaError_t dalloc(smpc_handle* h, T** p, size_t n) {
  cudaError_t e = cudaMalloc((void**)p, n * sizeof(T));
  if (e == cudaSuccess) { h->allocs.push_back(*p); e = cudaMemsetAsync(*p, 0, n * sizeof(T), h->stream); }
  return e;
}

// caller array -> device pointer (copy through the staging area when the caller is on the host)
struct In {
  const void* dev = nullptr;
};
int stage_reserve(smpc_handle* h, size_t bytes) {
  if (bytes <= h->stage_bytes) return 0;
  if (h->stage) cudaFree(h->stage);
  h->stage = nullptr; h->stage_bytes = 0;
  CK(h, cudaMalloc(&h->stage, bytes));
  h->stage_bytes = bytes;
  return 0;
}

int copy_in(smpc_handle* h, void* dst, const void* src, size_t bytes, int mem) {
  CK(h, cudaMemcpyAsync(dst, src, bytes, mem == SMPC_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, h->stream));
  if (mem == SMPC_HOST) CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}
int copy_out(smpc_handle* h, void* dst, const void* src, size_t bytes, int mem) {
  if (!dst) return 0;
  CK(h, cudaMemcpyAsync(dst, src, bytes, mem == SMPC_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
  if (mem == SMPC_HOST) CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int check_launch(smpc_handle* h, const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(h, SMPC_ERR_CUDA, what, e);
  return 0;
}

// mask pointer: NULL stays NULL (= all problems)
int mask_in(smpc_handle* h, const uint8_t* active, int mem, const uint8_t** out) {
  if (!active) { *out = nullptr; return 0; }
  if (mem == SMPC_DEVICE) { *out = active; return 0; }
  int rc = copy_in(h, h->act, active, (size_t)h->B, SMPC_HOST);
  *out = h->act;
  return rc;
}

// viability network on the rows selected by `mode`: strict fp64-accumulate kernel or the tensor-core kernel (nn_precision)
void run_mlp(smpc_handle* h, int B, int N, int mode, int n_flat, const double* xsrc, const uint8_t* act, const uint8_t* need, double* out11,
             bool want_grad) {
  LaunchCtx c = h->ctx();
  const int32_t* ridx = h->P.nn_rows == SMPC_NN_PARALLEL ? h->cand : h->r;      // stage index of the gated row
  if (h->P.nn_precision == SMPC_NN_TF32X3 && h->tc_pair) launch_mlp_tc2(c, h->dP, h->wtc, h->n_sm, B, N, mode, n_flat, xsrc, ridx, act, need, out11, want_grad);
  else if (h->P.nn_precision == SMPC_NN_TF32X3) launch_mlp_tc(c, h->dP, h->wtc, h->n_sm, B, N, mode, n_flat, xsrc, ridx, act, need, out11, want_grad);
  else launch_mlp(c, h->dP, h->w, B, N, mode, n_flat, xsrc, ridx, act, need, out11, want_grad);
}

// linearise + QP for the problems in `act` at the stored guess: AbstractController.solve (controller.py:136-167)
int solve_pipeline(smpc_handle* h, const double* x0_dev, const uint8_t* act) {
  LaunchCtx c = h->ctx();
  const int B = h->B, N = h->N;
  if (h->timed) cudaEventRecord(h->ev[0], h->stream);
  if (h->P.nn_rows != SMPC_NN_NONE) {
    const int mode = h->P.nn_rows == SMPC_NN_TERMINAL ? ROWS_TERMINAL : (h->P.nn_rows == SMPC_NN_EVERYWHERE ? ROWS_ALL : (h->P.nn_rows == SMPC_NN_PARALLEL ? ROWS_CAND : ROWS_RECEDING));
    run_mlp(h, B, N, mode, 0, h->xg, act, nullptr, h->nn11, true);
  }
  launch_linearize(c, h->dP, B, N, h->xg, h->ug, h->P.nn_rows == SMPC_NN_PARALLEL ? h->cand : h->r, act, h->nn11, h->ee_traj, h->n_traj, h->cur_step, QPCALL(h, qp_rec), h->qpf != nullptr);
  if (h->timed) cudaEventRecord(h->ev[1], h->stream);
  cudaError_t qe = h->qpf ? f32::launch_qp_solve(c, h->dP, h->qpf, x0_dev, h->r, act, h->xt, h->ut, h->status, h->qp_iter, h->qp_status, h->qp_res)
                          : f64::launch_qp_solve(c, h->dP, h->qp, x0_dev, h->r, act, h->xt, h->ut, h->status, h->qp_iter, h->qp_status, h->qp_res);
  if (qe != cudaSuccess) return fail(h, SMPC_ERR_CUDA, "QP solve", qe);
  h->solved = true;
  if (h->timed) cudaEventRecord(h->ev[2], h->stream);
  return check_launch(h, "solve pipeline");
}

// controller.step for the problems in `act` (device pointers)
int step_pipeline(smpc_handle* h, const double* x_dev, const uint8_t* act, double* u_dev, uint8_t* abort_dev) {
  LaunchCtx c = h->ctx();
  const int B = h->B, N = h->N;
  launch_prep(c, h->dP, B, N, h->xg, h->ug, act, h->P.controller != SMPC_CTRL_REAL_RECEDING);
  if (h->P.controller == SMPC_CTRL_PARALLEL) {
    // ParallelController.step (controller.py:614-640): one batched solve per candidate node n = N .. 1 for the problems that have
    // not reached n = N yet; the host reads one counter per candidate to stop early
    launch_par_begin(c, B, act, h->par_best, h->par_done, h->par_act, h->par_open);
    for (int n = N; n >= 1; --n) {
      launch_fill_i32(c, h->cand, B, n);
      int rc = solve_pipeline(h, x_dev, h->par_act);
      if (rc) return rc;
      run_mlp(h, B, N, ROWS_ALL, 0, h->xt, h->par_act, nullptr, h->scan11, false);
      launch_par_eval(c, h->dP, B, N, n, h->par_act, h->status, h->r, h->xt, h->ut, h->scan11, h->par_best, h->par_xt, h->par_ut, h->par_done,
                      h->par_act, h->par_open);
      CK(h, cudaMemcpyAsync(h->h_par_open, h->par_open, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
      CK(h, cudaStreamSynchronize(h->stream));
      if (*h->h_par_open == 0) break;
    }
    launch_par_post(c, h->dP, B, N, act, h->xg, h->ug, h->xt, h->ut, h->par_best, h->par_xt, h->par_ut, h->fails, h->r, h->x_viable, h->need_scan,
                    abort_dev, u_dev);
    launch_ctrl_post2(c, h->dP, B, N, act, h->xg, h->ug, h->xt, h->ut, h->fails, h->r, h->cur_step, h->need_scan, h->scan11, abort_dev, u_dev);
    if (h->timed) cudaEventRecord(h->ev[3], h->stream);
    return check_launch(h, "parallel controller step pipeline");
  }
  int rc = solve_pipeline(h, x_dev, act);
  if (rc) return rc;
  launch_ctrl_post1(c, h->dP, B, N, act, h->xg, h->ug, h->xt, h->status, h->fails, h->r, h->x_viable, h->need_scan, abort_dev, u_dev);
  if (h->P.controller == SMPC_CTRL_RECEDING || h->P.controller == SMPC_CTRL_REAL_RECEDING)
    run_mlp(h, B, N, ROWS_ALL, 0, h->xt, act, h->need_scan, h->scan11, false);
  launch_ctrl_post2(c, h->dP, B, N, act, h->xg, h->ug, h->xt, h->ut, h->fails, h->r, h->cur_step, h->need_scan, h->scan11, abort_dev, u_dev);
  if (h->timed) cudaEventRecord(h->ev[3], h->stream);
  return check_launch(h, "controller step pipeline");
}

// Stream capture (CUDA graphs, INTEGRATION.md).  *cap: the handle's stream is being captured.  A capture that has been invalidated is an
// error; a captured call must not read anything back on the host, so host arrays, the parallel controller (its early stop reads a
// counter), profiling / SMPC_QP_TRACE (timelines read on the host) and several tile groups are refused before anything is queued.
int capture_state(smpc_handle* h, const char* what, bool* cap) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  const cudaError_t e = cudaStreamIsCapturing(h->stream, &cs);
  if (e != cudaSuccess) return fail(h, SMPC_ERR_CUDA, what, e);
  if (cs == cudaStreamCaptureStatusInvalidated) {
    char buf[256];
    snprintf(buf, sizeof buf, "%s: the capture of the handle's stream has been invalidated", what);
    return fail(h, SMPC_ERR_CUDA, buf);
  }
  *cap = cs == cudaStreamCaptureStatusActive;
  return 0;
}
int capture_refuse(smpc_handle* h, const char* what, int mem, bool solves) {
  char buf[256];
  if (mem == SMPC_HOST) {
    snprintf(buf, sizeof buf, "%s: host arrays cannot be used in a stream capture (they need a synchronising copy); pass device pointers", what);
    return fail(h, SMPC_ERR_ARG, buf);
  }
  if (!solves) return 0;
  if (h->P.controller == SMPC_CTRL_PARALLEL) {
    snprintf(buf, sizeof buf, "%s: the parallel controller cannot be captured (its early stop reads a device counter on the host)", what);
    return fail(h, SMPC_ERR_UNSUPPORTED, buf);
  }
  if (QPCALL(h, qp_traced)) {
    snprintf(buf, sizeof buf, "%s: profiling / SMPC_QP_TRACE read the kernel timeline on the host and cannot be captured", what);
    return fail(h, SMPC_ERR_UNSUPPORTED, buf);
  }
  if (QPCALL(h, qp_groups) != 1) {
    snprintf(buf, sizeof buf, "%s: a QP solve over several tile groups (SMPC_QP_GROUPS) cannot be captured", what);
    return fail(h, SMPC_ERR_UNSUPPORTED, buf);
  }
  return 0;
}

void collect_times(smpc_handle* h, bool with_post) {
  float lin = 0, qp = 0, post = 0;
  cudaEventElapsedTime(&lin, h->ev[0], h->ev[1]);
  cudaEventElapsedTime(&qp, h->ev[1], h->ev[2]);
  if (with_post) cudaEventElapsedTime(&post, h->ev[2], h->ev[3]);
  h->times[0] = lin; h->times[1] = 0.0; h->times[2] = qp; h->times[3] = qp; h->times[4] = post; h->times[5] = 0.0;
  h->times[6] = lin + qp + post;
}

}  // namespace

extern "C" {

const char* smpc_version(void) { return "safe_mpc_b200 0.1.0 (sm_100a)"; }

const char* smpc_last_error(const smpc_handle_t* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int smpc_create(const smpc_problem_t* prob, int32_t batch, int32_t device, smpc_handle_t** out) {
  if (!prob || !out || batch <= 0) return fail(nullptr, SMPC_ERR_ARG, "smpc_create: bad arguments");
  if (prob->nq != SMPC_NQ || prob->n_pairs != SMPC_NPAIR || prob->N < 2 || prob->N > SMPC_MAX_N || prob->n_points > SMPC_MAX_POINTS)
    return fail(nullptr, SMPC_ERR_UNSUPPORTED, "smpc_create: unsupported dimensions (this build: nq=5, 6 capsule pairs, 2<=N<=128)");
  if (prob->nn_rows != SMPC_NN_NONE && !prob->nn_weights) return fail(nullptr, SMPC_ERR_ARG, "smpc_create: nn_rows set but nn_weights is NULL");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(nullptr, SMPC_ERR_CUDA, "smpc_create: no CUDA device (this engine has no CPU fallback)", e);
  if (device < 0 || device >= ndev) return fail(nullptr, SMPC_ERR_ARG, "smpc_create: bad device index");
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, SMPC_ERR_CUDA, "cudaSetDevice", e);
  smpc_handle* h = new smpc_handle;
  h->P = *prob;
  h->B = batch; h->N = prob->N; h->device = device;
  const int B = batch, N = prob->N;
#define CKC(call)                                                                                     \
  do {                                                                                                \
    cudaError_t e__ = (call);                                                                         \
    if (e__ != cudaSuccess) { fail(nullptr, SMPC_ERR_CUDA, #call, e__); smpc_destroy(h); return SMPC_ERR_CUDA; } \
  } while (0)
  CKC(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  for (auto& ev : h->ev) CKC(cudaEventCreate(&ev));
  CKC(mlp_prepare());
  CKC(linearize_prepare());
  // network weights: original + transposed copies of the two square layers
  if (prob->nn_weights) {
    const size_t np = SMPC_NN_NPARAM, sq = (size_t)SMPC_HID * SMPC_HID;
    CKC(dalloc(h, &h->dW, np + 2 * sq));
    std::vector<float> host(np + 2 * sq);
    std::memcpy(host.data(), prob->nn_weights, np * sizeof(float));
    const float* W1 = host.data();
    const float* b1 = W1 + SMPC_HID * SMPC_NX;
    const float* W2 = b1 + SMPC_HID;
    const float* b2 = W2 + sq;
    const float* W3 = b2 + SMPC_HID;
    float* W2t = host.data() + np;
    float* W3t = W2t + sq;
    for (int i = 0; i < SMPC_HID; ++i)
      for (int j = 0; j < SMPC_HID; ++j) { W2t[(size_t)j * SMPC_HID + i] = W2[(size_t)i * SMPC_HID + j]; W3t[(size_t)j * SMPC_HID + i] = W3[(size_t)i * SMPC_HID + j]; }
    CKC(cudaMemcpyAsync(h->dW, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CKC(cudaStreamSynchronize(h->stream));
    float* d = h->dW;
    h->w.W1 = d; d += SMPC_HID * SMPC_NX; h->w.b1 = d; d += SMPC_HID;
    h->w.W2 = d; d += sq; h->w.b2 = d; d += SMPC_HID;
    h->w.W3 = d; d += sq; h->w.b3 = d; d += SMPC_HID;
    h->w.W4 = d; d += SMPC_HID; h->w.b4 = d; d += 1;
    h->w.W2t = d; d += sq; h->w.W3t = d;
    if (prob->nn_precision == SMPC_NN_TF32X3) {
      cudaDeviceProp dp;
      CKC(cudaGetDeviceProperties(&dp, device));
      if (dp.major < 10) { fail(nullptr, SMPC_ERR_UNSUPPORTED, "smpc_create: nn_precision = SMPC_NN_TF32X3 needs tcgen05 (sm_100a)"); smpc_destroy(h); return SMPC_ERR_UNSUPPORTED; }
      h->n_sm = dp.multiProcessorCount;
      std::vector<float> packed(mlp_tc_packed_floats());
      mlp_tc_pack(W2, W3, packed.data());
      CKC(dalloc(h, &h->dWtc, packed.size()));
      CKC(cudaMemcpyAsync(h->dWtc, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
      CKC(cudaStreamSynchronize(h->stream));
      CKC(mlp_tc_prepare());
      std::vector<float> packed2(mlp_tc2_packed_floats());
      mlp_tc2_pack(W2, W3, packed2.data());
      CKC(dalloc(h, &h->dWtc2, packed2.size()));
      CKC(cudaMemcpyAsync(h->dWtc2, packed2.data(), packed2.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
      CKC(cudaStreamSynchronize(h->stream));
      CKC(mlp_tc2_prepare());
      if (const char* te = getenv("SMPC_MLP_TC")) h->tc_pair = strcmp(te, "pair") == 0;
      h->wtc = MlpTcWeights{h->w.W1, h->w.b1, h->w.b2, h->w.b3, h->w.W4, h->w.b4, h->dWtc, h->dWtc2};
    }
  }
  if (prob->precision != SMPC_PREC_F64 && prob->precision != SMPC_PREC_F32) {
    fail(nullptr, SMPC_ERR_ARG, "smpc_create: unknown precision"); smpc_destroy(h); return SMPC_ERR_ARG;
  }
  if (prob->nn_precision != SMPC_NN_STRICT && prob->nn_precision != SMPC_NN_TF32X3) {
    fail(nullptr, SMPC_ERR_ARG, "smpc_create: unknown nn_precision"); smpc_destroy(h); return SMPC_ERR_ARG;
  }
  CKC(dalloc(h, &h->dP, 1));
  {
    smpc_problem_t tmp = *prob;
    tmp.nn_weights = h->dW;
    CKC(cudaMemcpyAsync(h->dP, &tmp, sizeof tmp, cudaMemcpyHostToDevice, h->stream));
    CKC(cudaStreamSynchronize(h->stream));
  }
  const size_t nx = (size_t)B * (N + 1) * NX, nu = (size_t)B * N * NU, nst = (size_t)B * (N + 1);
  CKC(dalloc(h, &h->xg, nx)); CKC(dalloc(h, &h->ug, nu)); CKC(dalloc(h, &h->xt, nx)); CKC(dalloc(h, &h->ut, nu));
  CKC(dalloc(h, &h->plant_inertial, (size_t)B * NQ * 10)); CKC(dalloc(h, &h->tau_noise, (size_t)B * NU));
  CKC(dalloc(h, &h->x_viable, (size_t)B * NX));
  CKC(dalloc(h, &h->nn11, nst * NN_OUT));
  if (prob->controller == SMPC_CTRL_RECEDING || prob->controller == SMPC_CTRL_REAL_RECEDING || prob->controller == SMPC_CTRL_PARALLEL)
    CKC(dalloc(h, &h->scan11, nst * NN_OUT));
  CKC(dalloc(h, &h->cand, (size_t)B));
  if (prob->controller == SMPC_CTRL_PARALLEL) {
    if (prob->nn_rows != SMPC_NN_PARALLEL) { fail(nullptr, SMPC_ERR_ARG, "smpc_create: SMPC_CTRL_PARALLEL needs nn_rows = SMPC_NN_PARALLEL"); smpc_destroy(h); return SMPC_ERR_ARG; }
    CKC(dalloc(h, &h->par_best, (size_t)B)); CKC(dalloc(h, &h->par_done, (size_t)B)); CKC(dalloc(h, &h->par_act, (size_t)B));
    CKC(dalloc(h, &h->par_xt, nx)); CKC(dalloc(h, &h->par_ut, nu)); CKC(dalloc(h, &h->par_open, (size_t)1));
    CKC(cudaMallocHost((void**)&h->h_par_open, sizeof(int)));
  }
  {
    cudaError_t qe = cudaSuccess;
    if (prob->precision == SMPC_PREC_F32) h->qpf = f32::qp_create(B, N, prob->qp_iter_max, prob->qp_keep_slots != 0, h->stream, &qe);
    else h->qp = f64::qp_create(B, N, prob->qp_iter_max, prob->qp_keep_slots != 0, h->stream, &qe);
    if (!h->qp && !h->qpf) { fail(nullptr, SMPC_ERR_CUDA, "qp_create", qe); smpc_destroy(h); return SMPC_ERR_CUDA; }
  }
  CKC(dalloc(h, &h->qp_res, (size_t)B * 5));
  CKC(dalloc(h, &h->x_in, (size_t)B * NX)); CKC(dalloc(h, &h->u_out, (size_t)B * NU));
  CKC(dalloc(h, &h->fails, (size_t)B)); CKC(dalloc(h, &h->r, (size_t)B)); CKC(dalloc(h, &h->status, (size_t)B));
  CKC(dalloc(h, &h->qp_iter, (size_t)B)); CKC(dalloc(h, &h->qp_status, (size_t)B)); CKC(dalloc(h, &h->cur_step, (size_t)B));
  CKC(dalloc(h, &h->act, (size_t)B)); CKC(dalloc(h, &h->need_scan, (size_t)B)); CKC(dalloc(h, &h->abort_flag, (size_t)B));
  // defaults: plant = nominal model, r = N, status = 4 (controller.py:125)
  {
    std::vector<double> pin((size_t)B * NQ * 10);
    for (int b = 0; b < B; ++b) std::memcpy(&pin[(size_t)b * NQ * 10], prob->inertial, sizeof(double) * NQ * 10);
    CKC(cudaMemcpyAsync(h->plant_inertial, pin.data(), pin.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CKC(cudaStreamSynchronize(h->stream));
  }
  LaunchCtx c = h->ctx();
  launch_fill_i32(c, h->r, B, N);
  launch_fill_i32(c, h->cand, B, N);
  launch_fill_i32(c, h->status, B, 4);
  CKC(cudaStreamSynchronize(h->stream));
  CKC(cudaGetLastError());
#undef CKC
  *out = h;
  return SMPC_OK;
}

void smpc_destroy(smpc_handle_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->h_par_open) cudaFreeHost(h->h_par_open);
  for (void* p : h->allocs) cudaFree(p);
  f64::qp_destroy(h->qp);
  f32::qp_destroy(h->qpf);
  if (h->stage) cudaFree(h->stage);
  if (h->ee_traj) cudaFree(h->ee_traj);
  for (auto& ev : h->ev) if (ev) cudaEventDestroy(ev);
  if (h->stream && h->own_stream) cudaStreamDestroy(h->stream);
  delete h;
}

int smpc_set_plant_inertial(smpc_handle_t* h, const double* v, int32_t mem) { return copy_in(h, h->plant_inertial, v, sizeof(double) * h->B * NQ * 10, mem); }
int smpc_set_torque_noise(smpc_handle_t* h, const double* v, int32_t mem) { return copy_in(h, h->tau_noise, v, sizeof(double) * h->B * NU, mem); }

int smpc_set_ee_trajectory(smpc_handle_t* h, const double* traj, int32_t n, int32_t mem) {
  if (!h) return SMPC_ERR_ARG;
  if (n < 0 || (n > 0 && !traj)) return fail(h, SMPC_ERR_ARG, "smpc_set_ee_trajectory: n < 0 or missing array");
  if (cudaSetDevice(h->device) != cudaSuccess) return fail(h, SMPC_ERR_CUDA, "cudaSetDevice", cudaGetLastError());
  cudaStreamSynchronize(h->stream);                         // no solve may still read the array that is replaced
  if (h->ee_traj) { cudaFree(h->ee_traj); h->ee_traj = nullptr; }
  h->n_traj = 0;
  if (n == 0) return SMPC_OK;
  cudaError_t e = cudaMalloc((void**)&h->ee_traj, sizeof(double) * 3 * (size_t)n);
  if (e != cudaSuccess) return fail(h, SMPC_ERR_CUDA, "smpc_set_ee_trajectory: cudaMalloc", e);
  const int rc = copy_in(h, h->ee_traj, traj, sizeof(double) * 3 * (size_t)n, mem);
  if (rc) return rc;
  h->n_traj = n;
  return SMPC_OK;
}

int smpc_set_guess(smpc_handle_t* h, const double* xg, const double* ug, int32_t mem) {
  int rc = copy_in(h, h->xg, xg, sizeof(double) * h->B * (h->N + 1) * NX, mem);
  if (rc) return rc;
  rc = copy_in(h, h->ug, ug, sizeof(double) * h->B * h->N * NU, mem);
  if (rc) return rc;
  launch_set_xviable_from_guess(h->ctx(), h->B, h->N, h->xg, h->x_viable);
  return check_launch(h, "set_guess");
}
int smpc_get_guess(smpc_handle_t* h, double* xg, double* ug, int32_t mem) {
  int rc = copy_out(h, xg, h->xg, sizeof(double) * h->B * (h->N + 1) * NX, mem);
  return rc ? rc : copy_out(h, ug, h->ug, sizeof(double) * h->B * h->N * NU, mem);
}
int smpc_get_temp(smpc_handle_t* h, double* xt, double* ut, int32_t mem) {
  int rc = copy_out(h, xt, h->xt, sizeof(double) * h->B * (h->N + 1) * NX, mem);
  return rc ? rc : copy_out(h, ut, h->ut, sizeof(double) * h->B * h->N * NU, mem);
}
int smpc_reset_controller(smpc_handle_t* h) {
  LaunchCtx c = h->ctx();
  launch_fill_i32(c, h->fails, h->B, 0);
  launch_fill_i32(c, h->r, h->B, h->N);
  launch_fill_i32(c, h->cur_step, h->B, 0);
  return check_launch(h, "reset_controller");
}

int smpc_rti_solve(smpc_handle_t* h, const double* x0, const uint8_t* active, int32_t* status, int32_t mem) {
  if (!x0) return fail(h, SMPC_ERR_ARG, "smpc_rti_solve: x0 is NULL");
  bool cap = false;
  int rc = capture_state(h, "smpc_rti_solve", &cap);
  if (!rc && cap) rc = capture_refuse(h, "smpc_rti_solve", mem, true);
  if (rc) return rc;
  const uint8_t* act = nullptr;
  rc = mask_in(h, active, mem, &act);
  if (rc) return rc;
  const double* xd = x0;
  if (mem == SMPC_HOST) { rc = copy_in(h, h->x_in, x0, sizeof(double) * h->B * NX, mem); if (rc) return rc; xd = h->x_in; }
  h->timed = !cap;                   // (a replay of a captured step records no times: smpc_get_times keeps the last eager step)
  rc = solve_pipeline(h, xd, act);
  if (rc) return rc;
  if (!cap) h->times_pending = 1;
  return copy_out(h, status, h->status, sizeof(int32_t) * h->B, mem);
}

int smpc_controller_step(smpc_handle_t* h, const double* x, const uint8_t* active, double* u, uint8_t* abort_flag, int32_t mem) {
  if (!x || !u) return fail(h, SMPC_ERR_ARG, "smpc_controller_step: x or u is NULL");
  bool cap = false;
  int rc = capture_state(h, "smpc_controller_step", &cap);
  if (!rc && cap) rc = capture_refuse(h, "smpc_controller_step", mem, true);
  if (rc) return rc;
  const uint8_t* act = nullptr;
  rc = mask_in(h, active, mem, &act);
  if (rc) return rc;
  const double* xd = x;
  double* ud = u;
  uint8_t* ad = abort_flag;
  if (mem == SMPC_HOST) {
    rc = copy_in(h, h->x_in, x, sizeof(double) * h->B * NX, mem); if (rc) return rc;
    rc = copy_in(h, h->u_out, u, sizeof(double) * h->B * NU, mem); if (rc) return rc;   // inactive problems keep the caller's values
    xd = h->x_in; ud = h->u_out; ad = h->abort_flag;
  } else if (!ad) ad = h->abort_flag;
  h->timed = !cap;
  rc = step_pipeline(h, xd, act, ud, ad);
  if (rc) return rc;
  if (!cap) h->times_pending = 2;
  if (mem == SMPC_HOST) {
    rc = copy_out(h, u, h->u_out, sizeof(double) * h->B * NU, mem); if (rc) return rc;
    rc = copy_out(h, abort_flag, h->abort_flag, (size_t)h->B, mem);
  }
  return rc;
}

int smpc_plant_step(smpc_handle_t* h, const double* x, const double* u, double* xn, double* a, int32_t mem) {
  const size_t bx = sizeof(double) * h->B * NX, bu = sizeof(double) * h->B * NU;
  bool cap = false;
  int rc0 = capture_state(h, "smpc_plant_step", &cap);
  if (!rc0 && cap) rc0 = capture_refuse(h, "smpc_plant_step", mem, false);
  if (rc0) return rc0;
  if (mem == SMPC_DEVICE) {
    launch_plant(h->ctx(), h->dP, h->B, h->plant_inertial, h->tau_noise, x, u, nullptr, xn, a);
    return check_launch(h, "plant_step");
  }
  int rc = stage_reserve(h, 2 * bx + 2 * bu); if (rc) return rc;
  char* s = (char*)h->stage;
  double *dx = (double*)s, *du = (double*)(s + bx), *dxn = (double*)(s + bx + bu), *da = (double*)(s + 2 * bx + bu);
  rc = copy_in(h, dx, x, bx, mem); if (rc) return rc;
  rc = copy_in(h, du, u, bu, mem); if (rc) return rc;
  launch_plant(h->ctx(), h->dP, h->B, h->plant_inertial, h->tau_noise, dx, du, nullptr, dxn, da);
  rc = check_launch(h, "plant_step"); if (rc) return rc;
  rc = copy_out(h, xn, dxn, bx, mem); if (rc) return rc;
  return copy_out(h, a, da, bu, mem);
}

int smpc_tau(smpc_handle_t* h, int32_t n, const double* x, const double* u, double* tau, int32_t mem) {
  if (n <= 0) return SMPC_OK;
  const size_t bx = sizeof(double) * n * NX, bu = sizeof(double) * n * NU;
  if (mem == SMPC_DEVICE) { launch_tau(h->ctx(), h->dP, n, x, u, tau); return check_launch(h, "tau"); }
  int rc = stage_reserve(h, bx + 2 * bu); if (rc) return rc;
  char* s = (char*)h->stage;
  rc = copy_in(h, s, x, bx, mem); if (rc) return rc;
  rc = copy_in(h, s + bx, u, bu, mem); if (rc) return rc;
  launch_tau(h->ctx(), h->dP, n, (double*)s, (double*)(s + bx), (double*)(s + bx + bu));
  rc = check_launch(h, "tau"); if (rc) return rc;
  return copy_out(h, tau, s + bx + bu, bu, mem);
}

int smpc_rk4_sens(smpc_handle_t* h, int32_t n, const double* x, const double* tau, double dt, double* x_next, double* A, double* B, int32_t mem) {
  if (n <= 0) return SMPC_OK;
  if (!x || !tau || !x_next || !(dt > 0.0)) return fail(h, SMPC_ERR_ARG, "rk4_sens: x, tau, x_next must be given and dt > 0");
  const size_t bx = sizeof(double) * n * NX, bu = sizeof(double) * n * NU, ba = A ? bx * NX : 0, bb = B ? bx * NU : 0;
  if (mem == SMPC_DEVICE) { launch_rk4_sens(h->ctx(), h->dP, n, dt, x, tau, x_next, A, B); return check_launch(h, "rk4_sens"); }
  int rc = stage_reserve(h, 2 * bx + bu + ba + bb); if (rc) return rc;
  char* s = (char*)h->stage;
  double *dx = (double*)s, *dt_ = (double*)(s + bx), *dn = (double*)(s + bx + bu), *dA = A ? (double*)(s + 2 * bx + bu) : nullptr,
         *dB = B ? (double*)(s + 2 * bx + bu + ba) : nullptr;
  rc = copy_in(h, dx, x, bx, mem); if (rc) return rc;
  rc = copy_in(h, dt_, tau, bu, mem); if (rc) return rc;
  launch_rk4_sens(h->ctx(), h->dP, n, dt, dx, dt_, dn, dA, dB);
  rc = check_launch(h, "rk4_sens"); if (rc) return rc;
  rc = copy_out(h, x_next, dn, bx, mem); if (rc) return rc;
  if (A) { rc = copy_out(h, A, dA, ba, mem); if (rc) return rc; }
  if (B) { rc = copy_out(h, B, dB, bb, mem); if (rc) return rc; }
  return SMPC_OK;
}

int smpc_kinematics(smpc_handle_t* h, int32_t n, const double* x, double* ee, double* dist, int32_t mem) {
  if (n <= 0) return SMPC_OK;
  const size_t bx = sizeof(double) * n * NX, be = sizeof(double) * n * 3, bd = sizeof(double) * n * NPAIR;
  if (mem == SMPC_DEVICE) { launch_kin(h->ctx(), h->dP, n, x, ee, dist); return check_launch(h, "kinematics"); }
  int rc = stage_reserve(h, bx + be + bd); if (rc) return rc;
  char* s = (char*)h->stage;
  rc = copy_in(h, s, x, bx, mem); if (rc) return rc;
  launch_kin(h->ctx(), h->dP, n, (double*)s, (double*)(s + bx), (double*)(s + bx + be));
  rc = check_launch(h, "kinematics"); if (rc) return rc;
  rc = copy_out(h, ee, s + bx, be, mem); if (rc) return rc;
  return copy_out(h, dist, s + bx + be, bd, mem);
}

int smpc_nn_constraint(smpc_handle_t* h, int32_t n, const double* x, double* cval, double* grad, int32_t mem) {
  if (!h->dW) return fail(h, SMPC_ERR_ARG, "smpc_nn_constraint: this handle has no viability network");
  if (n <= 0) return SMPC_OK;
  const size_t bx = sizeof(double) * n * NX, bo = sizeof(double) * n * NN_OUT;
  int rc = stage_reserve(h, bx + bo + sizeof(double) * n * (NX + 1)); if (rc) return rc;
  char* s = (char*)h->stage;
  const double* xd = x;
  if (mem == SMPC_HOST) { rc = copy_in(h, s, x, bx, mem); if (rc) return rc; xd = (double*)s; }
  double* o11 = (double*)(s + bx);
  run_mlp(h, n, 0, ROWS_FLAT, n, xd, nullptr, nullptr, o11, true);
  rc = check_launch(h, "nn_constraint"); if (rc) return rc;
  // de-interleave [n][11] -> c[n], grad[n][10]
  double* dc = (double*)(s + bx + bo);
  double* dg = dc + n;
  CK(h, cudaMemcpy2DAsync(dc, sizeof(double), o11, sizeof(double) * NN_OUT, sizeof(double), n, cudaMemcpyDeviceToDevice, h->stream));
  CK(h, cudaMemcpy2DAsync(dg, sizeof(double) * NX, o11 + 1, sizeof(double) * NN_OUT, sizeof(double) * NX, n, cudaMemcpyDeviceToDevice, h->stream));
  rc = copy_out(h, cval, dc, sizeof(double) * n, mem); if (rc) return rc;
  return copy_out(h, grad, dg, sizeof(double) * n * NX, mem);
}

static int slots_intact(smpc_handle_t* h, const char* what) {
  if (QPCALL(h, qp_compactions) == 0) return 0;
  char buf[256];
  snprintf(buf, sizeof buf, "%s: the last solve compacted its slots (the stage records / iterates of the finished problems were reused); "
                            "create the handle with smpc_problem_t::qp_keep_slots = 1 (or SMPC_QP_COMPACT=0) to keep them", what);
  return fail(h, SMPC_ERR_UNSUPPORTED, buf);
}

int smpc_get_lin(smpc_handle_t* h, double* lin, int32_t mem) {
  if (int rc0 = slots_intact(h, "smpc_get_lin")) return rc0;
  const size_t bytes = sizeof(double) * h->B * (h->N + 1) * REC;
  if (mem == SMPC_DEVICE) { if (h->qpf) f32::launch_rec_untile(h->ctx(), h->qpf, lin); else f64::launch_rec_untile(h->ctx(), h->qp, lin); return check_launch(h, "get_lin"); }
  int rc = stage_reserve(h, bytes); if (rc) return rc;
  if (h->qpf) f32::launch_rec_untile(h->ctx(), h->qpf, (double*)h->stage);      // records are kept tile-interleaved; hand them back as [B][N+1][REC]
  else f64::launch_rec_untile(h->ctx(), h->qp, (double*)h->stage);
  rc = check_launch(h, "get_lin"); if (rc) return rc;
  return copy_out(h, lin, h->stage, bytes, mem);
}

int smpc_get_qp(smpc_handle_t* h, double* dz, double* pi, double* lam, double* t, int32_t mem) {
  const size_t nst = (size_t)h->B * (h->N + 1);
  const size_t b1 = sizeof(double) * nst * 15, b2 = sizeof(double) * h->B * h->N * 10, b3 = sizeof(double) * nst * SMPC_QP_NC;
  if (!h->solved) return fail(h, SMPC_ERR_ARG, "smpc_get_qp: no smpc_rti_solve / smpc_controller_step yet");
  if (int rc0 = slots_intact(h, "smpc_get_qp")) return rc0;
  int rc = stage_reserve(h, b1 + b2 + 2 * b3); if (rc) return rc;
  char* s = (char*)h->stage;
  // the final iterate of every problem stays in the solver's ping-pong buffers until the next solve
  if (h->qpf) f32::launch_dump_qp(h->ctx(), h->dP, h->qpf, (double*)s, (double*)(s + b1), (double*)(s + b1 + b2), (double*)(s + b1 + b2 + b3));
  else f64::launch_dump_qp(h->ctx(), h->dP, h->qp, (double*)s, (double*)(s + b1), (double*)(s + b1 + b2), (double*)(s + b1 + b2 + b3));
  rc = check_launch(h, "get_qp"); if (rc) return rc;
  rc = copy_out(h, dz, s, b1, mem); if (rc) return rc;
  rc = copy_out(h, pi, s + b1, b2, mem); if (rc) return rc;
  rc = copy_out(h, lam, s + b1 + b2, b3, mem); if (rc) return rc;
  return copy_out(h, t, s + b1 + b2 + b3, b3, mem);
}

static int32_t* state_ptr(smpc_handle_t* h, int32_t f) {
  switch (f) {
    case SMPC_STATE_FAILS: return h->fails;
    case SMPC_STATE_R: return h->r;
    case SMPC_STATE_STATUS: return h->status;
    case SMPC_STATE_QP_ITER: return h->qp_iter;
    case SMPC_STATE_QP_STATUS: return h->qp_status;
  }
  return nullptr;
}
int smpc_get_state_i32(smpc_handle_t* h, int32_t f, int32_t* out, int32_t mem) {
  int32_t* p = state_ptr(h, f);
  if (!p) return fail(h, SMPC_ERR_ARG, "smpc_get_state_i32: unknown field");
  return copy_out(h, out, p, sizeof(int32_t) * h->B, mem);
}
int smpc_set_state_i32(smpc_handle_t* h, int32_t f, const int32_t* in, int32_t mem) {
  int32_t* p = state_ptr(h, f);
  if (!p) return fail(h, SMPC_ERR_ARG, "smpc_set_state_i32: unknown field");
  return copy_in(h, p, in, sizeof(int32_t) * h->B, mem);
}
int smpc_get_qp_residuals(smpc_handle_t* h, double* res5, int32_t mem) { return copy_out(h, res5, h->qp_res, sizeof(double) * h->B * 5, mem); }
int smpc_get_x_viable(smpc_handle_t* h, double* xv, int32_t mem) { return copy_out(h, xv, h->x_viable, sizeof(double) * h->B * NX, mem); }

int smpc_set_profiling(smpc_handle_t* h, int32_t enable) { QPCALL(h, qp_set_profiling, enable != 0); return SMPC_OK; }
int smpc_get_profile(smpc_handle_t* h, double* ms, int32_t* count, double* span_ms, int32_t* iterations) {
  if (!ms || !count || !span_ms || !iterations) return fail(h, SMPC_ERR_ARG, "smpc_get_profile: NULL output");
  QPCALL(h, qp_get_profile, ms, count, span_ms);
  *iterations = QPCALL(h, qp_last_iterations);
  return SMPC_OK;
}
int smpc_get_times(smpc_handle_t* h, double* out7) {
  if (h->times_pending) {
    CK(h, cudaStreamSynchronize(h->stream));
    collect_times(h, h->times_pending == 2);
    h->times_pending = 0;
  }
  for (int i = 0; i < 7; ++i) out7[i] = h->times[i];
  return SMPC_OK;
}
int64_t smpc_launch_count(const smpc_handle_t* h) { return h->launches; }
void* smpc_stream(smpc_handle_t* h) { return (void*)h->stream; }
int smpc_set_stream(smpc_handle_t* h, void* stream) {
  if (!h) return SMPC_ERR_ARG;
  if (cudaSetDevice(h->device) != cudaSuccess) return fail(h, SMPC_ERR_CUDA, "cudaSetDevice", cudaGetLastError());
  CK(h, cudaStreamSynchronize(h->stream));                  // everything queued so far is finished before the stream changes
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  if (stream) { h->stream = (cudaStream_t)stream; h->own_stream = false; }
  else { h->own_stream = true; CK(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); }
  return SMPC_OK;
}
int smpc_sync(smpc_handle_t* h) { CK(h, cudaStreamSynchronize(h->stream)); return check_launch(h, "sync"); }

// ------------------------------------------------------------------------------------------------ closed loop
int smpc_sim_create(smpc_handle_t* c, smpc_handle_t* bk, int32_t n_steps, smpc_sim_t** out) {
  if (!c || !bk || !out || n_steps <= 0 || c->B != bk->B || c->device != bk->device) return fail(c, SMPC_ERR_ARG, "smpc_sim_create: bad arguments");
  smpc_sim* s = new smpc_sim;
  s->c = c; s->bk = bk; s->device = c->device;
  SimDev& d = s->d;
  const int B = c->B, Nb = bk->N;
  d.B = B; d.N = c->N; d.Nb = Nb; d.n_steps = n_steps;
#define CKS(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { fail(c, SMPC_ERR_CUDA, #call, e__); s->allocs.insert(s->allocs.end(), c->allocs.begin() + n_before, c->allocs.end()); c->allocs.resize(n_before); smpc_sim_destroy(s); return SMPC_ERR_CUDA; } } while (0)
  const size_t n_before = c->allocs.size();      // dalloc registers with the handle; the buffers of the closed loop move to the sim object below
  CKS(dalloc(c, &d.x, (size_t)B * NX));
  CKS(dalloc(c, &d.xlog, (size_t)B * (n_steps + 1) * NX));
  CKS(dalloc(c, &d.ulog, (size_t)B * n_steps * NU));
  CKS(dalloc(c, &d.x_abort, (size_t)B * (Nb + 1) * NX));
  CKS(dalloc(c, &d.u_abort, (size_t)B * Nb * NU));
  CKS(dalloc(c, &d.xv_first, (size_t)B * NX));
  CKS(dalloc(c, &d.u_ctrl, (size_t)B * NU));
  CKS(dalloc(c, &d.u, (size_t)B * NU));
  CKS(dalloc(c, &d.mode, (size_t)B)); CKS(dalloc(c, &d.ja, (size_t)B)); CKS(dalloc(c, &d.outcome, (size_t)B));
  CKS(dalloc(c, &d.need_ctrl, (size_t)B)); CKS(dalloc(c, &d.need_backup, (size_t)B)); CKS(dalloc(c, &d.abort_flag, (size_t)B));
  CKS(dalloc(c, &d.live, (size_t)B));
  CKS(dalloc(c, &d.counters, (size_t)SIM_NCOUNTERS));
  CKS(cudaStreamCreateWithFlags(&s->body, cudaStreamNonBlocking));
  CKS(cudaMallocHost((void**)&s->h_requests, sizeof(unsigned long long)));
  CKS(dalloc(c, &s->outcome_tmp, (size_t)B));
#undef CKS
  s->allocs.assign(c->allocs.begin() + n_before, c->allocs.end());
  c->allocs.resize(n_before);
  *out = s;
  return SMPC_OK;
}
void smpc_sim_destroy(smpc_sim_t* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  cudaDeviceSynchronize();          // (the handles may already be gone: do not touch them)
  for (void* p : s->allocs) cudaFree(p);
  if (s->h_requests) cudaFreeHost(s->h_requests);
  if (s->body) cudaStreamDestroy(s->body);
  delete s;
}

int smpc_sim_reset(smpc_sim_t* s, const double* x_init, int32_t mem) {
  smpc_handle* c = s->c;
  SimDev& d = s->d;
  const int B = d.B;
  const double nan = __builtin_nan("");
  LaunchCtx lc = c->ctx();
  launch_fill_f64(lc, d.xlog, (size_t)B * (d.n_steps + 1) * NX, nan);
  launch_fill_f64(lc, d.ulog, (size_t)B * d.n_steps * NU, nan);
  launch_fill_f64(lc, d.xv_first, (size_t)B * NX, nan);
  launch_fill_i32(lc, d.mode, B, 0); launch_fill_i32(lc, d.ja, B, 0); launch_fill_i32(lc, d.outcome, B, 0);
  CK(c, cudaMemsetAsync(d.counters, 0, SIM_NCOUNTERS * sizeof(unsigned long long), c->stream));
  s->requests_seen = 0;
  int rc = copy_in(c, d.x, x_init, sizeof(double) * B * NX, mem); if (rc) return rc;
  CK(c, cudaMemcpy2DAsync(d.xlog, sizeof(double) * (d.n_steps + 1) * NX, d.x, sizeof(double) * NX, sizeof(double) * NX, B, cudaMemcpyDeviceToDevice, c->stream));
  s->j = 0;
  return check_launch(c, "sim_reset");
}

// The backup solve of a captured step: a one-thread kernel sets the condition (some problem asked for a backup solve in this step), and
// the body of a conditional IF node -- captured on s->body, with the backup handle launching there -- holds the backup pipeline, whose
// QP solve adds its own WHILE node inside (qp.cu).  The caller's stream continues after the IF node.
static int captured_backup(smpc_sim* s) {
  smpc_handle* c = s->c;
  smpc_handle* bk = s->bk;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaGraph_t graph = nullptr;
  const cudaGraphNode_t* deps = nullptr;
  size_t n_deps = 0;
  cudaGraphConditionalHandle cond = 0;
  CK(c, cudaStreamGetCaptureInfo(c->stream, &cs, nullptr, &graph, &deps, &n_deps));
  CK(c, cudaGraphConditionalHandleCreate(&cond, graph, 0, 0));     // (no default: the kernel below sets it on every launch)
  launch_sim_backup_cond(c->ctx(), s->d, cond);
  CK(c, cudaGetLastError());
  CK(c, cudaStreamGetCaptureInfo(c->stream, &cs, nullptr, &graph, &deps, &n_deps));
  cudaGraphNodeParams np = {};
  np.type = cudaGraphNodeTypeConditional;
  np.conditional.handle = cond;
  np.conditional.type = cudaGraphCondTypeIf;
  np.conditional.size = 1;
  cudaGraphNode_t node = nullptr;
  CK(c, cudaGraphAddNode(&node, graph, deps, n_deps, &np));
  // (from here on a failure leaves the capture with an incomplete node: the error is returned and the capture must be discarded)
  CK(c, cudaStreamUpdateCaptureDependencies(c->stream, &node, 1, cudaStreamSetCaptureDependencies));
  CK(c, cudaStreamBeginCaptureToGraph(s->body, np.conditional.phGraph_out[0], nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
  bk->stream = s->body;
  int rc = solve_pipeline(bk, c->x_viable, s->d.need_backup);   // safe_ocp.solve(x_viable), one RTI (mpc.py:177)
  bk->stream = c->stream;
  cudaGraph_t captured = nullptr;
  const cudaError_t e = cudaStreamEndCapture(s->body, &captured);   // (the body graph belongs to the node)
  if (rc) { c->err = bk->err; return rc; }
  if (e != cudaSuccess) return fail(c, SMPC_ERR_CUDA, "smpc_sim_step: capture of the backup solve", e);
  return 0;
}

int smpc_sim_step(smpc_sim_t* s) {
  smpc_handle* c = s->c;
  smpc_handle* bk = s->bk;
  SimDev& d = s->d;
  if (s->j >= d.n_steps) return fail(c, SMPC_ERR_ARG, "smpc_sim_step: past n_steps");
  bool cap = false;
  int rc = capture_state(c, "smpc_sim_step", &cap);
  if (!rc && cap) rc = capture_refuse(c, "smpc_sim_step", SMPC_DEVICE, true);
  if (!rc && cap && (rc = capture_refuse(bk, "smpc_sim_step (backup controller)", SMPC_DEVICE, true))) c->err = bk->err;
  if (rc) return rc;
  // both handles launch on the main controller's stream so that the step is one ordered sequence
  LaunchCtx lc = c->ctx();
  cudaStream_t bk_stream = bk->stream;
  bk->stream = c->stream;
  // captured: the step index and the backup decision live on the device (sim_pre / sim_post / sim_backup_cond in kernels.cu)
  launch_sim_pre(lc, d, c->dP, cap ? -1 : s->j);
  c->timed = !cap; bk->timed = false;           // the main controller's step is timed (smpc_get_times = controller.getTime(), mpc.py:239)
  rc = step_pipeline(c, d.x, d.need_ctrl, d.u_ctrl, d.abort_flag);
  if (!cap) c->times_pending = 2;
  if (!rc && cap) {
    launch_sim_mid(lc, d, c->x_viable, bk->xg, bk->ug, c->qp_iter);
    rc = captured_backup(s);                      // conditional IF node around the backup pipeline
  } else if (!rc) {
    launch_sim_mid(lc, d, c->x_viable, bk->xg, bk->ug, c->qp_iter);
    // the backup OCP is solved only in a step in which some problem aborted (mpc.py:168-177): one 8-byte read-back decides, instead of
    // an empty linearisation + QP launch sequence in every step (the host has waited for the main solve's counters anyway)
    cudaError_t e = cudaMemcpyAsync(s->h_requests, d.counters + 4, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = fail(c, SMPC_ERR_CUDA, "smpc_sim_step: backup request read-back", e);
    else if (*s->h_requests != s->requests_seen) {
      s->requests_seen = *s->h_requests;
      rc = solve_pipeline(bk, c->x_viable, d.need_backup);   // safe_ocp.solve(x_viable), one RTI (mpc.py:177)
    }
  }
  if (!rc) {
    launch_sim_post(lc, d, c->dP, cap ? -1 : s->j, bk->status, bk->xt, bk->ut, c->plant_inertial, c->tau_noise, bk->qp_iter);
    rc = check_launch(c, "sim_step");
  }
  bk->stream = bk_stream;                        // (restored on every path)
  if (!cap) s->j += 1;                           // (a captured step advances the device-side index on every replay)
  return rc;
}
int smpc_sim_run(smpc_sim_t* s, int32_t n) {
  for (int i = 0; i < n; ++i) { int rc = smpc_sim_step(s); if (rc) return rc; }
  return SMPC_OK;
}
int smpc_sim_get_outcome(smpc_sim_t* s, int32_t* out, int32_t mem) {
  launch_sim_outcome(s->c->ctx(), s->d, s->c->dP, s->outcome_tmp);
  int rc = check_launch(s->c, "sim_outcome"); if (rc) return rc;
  return copy_out(s->c, out, s->outcome_tmp, sizeof(int32_t) * s->d.B, mem);
}
int smpc_sim_get_log(smpc_sim_t* s, double* x, double* u, int32_t mem) {
  int rc = copy_out(s->c, x, s->d.xlog, sizeof(double) * s->d.B * (s->d.n_steps + 1) * NX, mem);
  return rc ? rc : copy_out(s->c, u, s->d.ulog, sizeof(double) * s->d.B * s->d.n_steps * NU, mem);
}
int smpc_sim_get_x_viable(smpc_sim_t* s, double* xv, int32_t mem) { return copy_out(s->c, xv, s->d.xv_first, sizeof(double) * s->d.B * NX, mem); }
int smpc_sim_get_counters(smpc_sim_t* s, int64_t* out4) {
  unsigned long long v[4];
  CK(s->c, cudaMemcpyAsync(v, s->d.counters, sizeof v, cudaMemcpyDeviceToHost, s->c->stream));
  CK(s->c, cudaStreamSynchronize(s->c->stream));
  for (int i = 0; i < 4; ++i) out4[i] = (int64_t)v[i];
  return SMPC_OK;
}

}  // extern "C"
