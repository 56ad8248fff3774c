// Kernels around the QP: warm-start correction, viability network, stage linearisation, controller state machines,
// plant step and the closed-loop bookkeeping.  Reference semantics are cited per kernel.
#include <cstdlib>
#include <cstring>

#include "engine.cuh"

namespace smpc {

#define GRID1D(n, t) (((n) + (t)-1) / (t))

// ----------------------------------------------------------------------------------------------------------------
// guessCorrection (reference controller.py:226-231): roll the guess forward with the double integrator
// ----------------------------------------------------------------------------------------------------------------
__global__ void prep_kernel(const smpc_problem_t* __restrict__ dP, int B, int N, double* xg, const double* __restrict__ ug,
                            const uint8_t* __restrict__ act, int correct) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B || (act && !act[b])) return;
  if (!correct) return;
  const double dt = dP->dt;
  double* x = xg + (size_t)b * (N + 1) * NX;
  const double* u = ug + (size_t)b * N * NU;
  double cur[NX];
#pragma unroll
  for (int i = 0; i < NX; ++i) cur[i] = x[i];
  for (int k = 0; k < N; ++k) {
    double nx[NX];
    f_disc(dt, cur, u + k * NU, nx);
#pragma unroll
    for (int i = 0; i < NX; ++i) { cur[i] = nx[i]; x[(k + 1) * NX + i] = nx[i]; }
  }
}
void launch_prep(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, double* xg, const double* ug, const uint8_t* act, bool correct) {
  prep_kernel<<<GRID1D(B, 128), 128, 0, c.stream>>>(dP, B, N, xg, ug, act, correct ? 1 : 0);
  ++*c.launches;
}

// ----------------------------------------------------------------------------------------------------------------
// Viability network, strict mode: fp32 weights, fp64 accumulation on the FP64 pipe (value + input gradient).
// NeuralNetwork / NetSafeSet of reference safe_set.py:26-43,71-104.  One CTA evaluates MLP_R rows; thread j owns
// hidden unit j of every layer, activations of the tile live in shared memory, weights stream from L2.
// ----------------------------------------------------------------------------------------------------------------
constexpr int MLP_R = 16;
constexpr int HID = SMPC_HID;

__global__ void __launch_bounds__(HID)
mlp_kernel(const smpc_problem_t* __restrict__ dP, MlpWeights w, int B, int N, int rows_mode, int n_rows, const double* __restrict__ xsrc,
           const int32_t* __restrict__ r, const uint8_t* __restrict__ act, const uint8_t* __restrict__ need, double* out11, int want_grad) {
  extern __shared__ double sm[];
  double* A0 = sm;                       // [R][HID]
  double* A1 = A0 + MLP_R * HID;         // [R][HID]
  double* D1 = A1 + MLP_R * HID;
  double* D2 = D1 + MLP_R * HID;
  double* D3 = D2 + MLP_R * HID;
  double* IN = D3 + MLP_R * HID;         // [R][10]
  double* NRM = IN + MLP_R * NX;         // [R]
  double* Y = NRM + MLP_R;               // [R]
  double* GIN = Y + MLP_R;               // [R][10]
  __shared__ int rowb[MLP_R], rowk[MLP_R], valid[MLP_R];
  const smpc_problem_t& P = *dP;
  const int j = threadIdx.x;
  const int row0 = blockIdx.x * MLP_R;
  if (j < MLP_R) {
    int b = 0, k = 0;
    const int i = row0 + j;
    const bool v = i < n_rows && mlp_row(rows_mode, i, B, N, r, act, need, b, k);
    valid[j] = v; rowb[j] = b; rowk[j] = k;
    double in[NX], nrm = 1.0;
    if (v) {
      const double* x = (rows_mode == ROWS_FLAT) ? xsrc + (size_t)b * NX : xsrc + ((size_t)b * (N + 1) + k) * NX;
      nn_input(P, x, in, &nrm);
    } else {
#pragma unroll
      for (int q = 0; q < NX; ++q) in[q] = 0.0;
    }
#pragma unroll
    for (int q = 0; q < NX; ++q) IN[j * NX + q] = in[q];
    NRM[j] = nrm;
  }
  __syncthreads();
  int any = 0;
  for (int q = 0; q < MLP_R; ++q) any |= valid[q];
  if (!any) return;
  double acc[MLP_R];
  // ---- layer 1 ----
  {
    const double bias = w.b1[j];
#pragma unroll
    for (int q = 0; q < MLP_R; ++q) acc[q] = bias;
    for (int k = 0; k < NX; ++k) {
      const double wv = w.W1[j * NX + k];
#pragma unroll
      for (int q = 0; q < MLP_R; ++q) acc[q] += wv * IN[q * NX + k];
    }
#pragma unroll
    for (int q = 0; q < MLP_R; ++q) { double d; A0[q * HID + j] = gelu_tanh(acc[q], &d); D1[q * HID + j] = d; }
  }
  __syncthreads();
  // ---- layers 2, 3 ----
#pragma unroll 1
  for (int layer = 0; layer < 2; ++layer) {
    const float* Wt = layer == 0 ? w.W2t : w.W3t;
    const double bias = layer == 0 ? w.b2[j] : w.b3[j];
    const double* Ain = layer == 0 ? A0 : A1;
    double* Aout = layer == 0 ? A1 : A0;
    double* Dout = layer == 0 ? D2 : D3;
#pragma unroll
    for (int q = 0; q < MLP_R; ++q) acc[q] = bias;
#pragma unroll 4
    for (int k = 0; k < HID; ++k) {
      const double wv = Wt[k * HID + j];
#pragma unroll
      for (int q = 0; q < MLP_R; ++q) acc[q] += wv * Ain[q * HID + k];
    }
#pragma unroll
    for (int q = 0; q < MLP_R; ++q) { double d; Aout[q * HID + j] = gelu_tanh(acc[q], &d); Dout[q * HID + j] = d; }
    __syncthreads();
  }
  // activations of layer 3 are in A0.  output: y = b4 + sum_j W4[j] a3[j]   (sequential in j, like the reference loop)
  if (j < MLP_R) {
    double y = w.b4[0];
    for (int k = 0; k < HID; ++k) y += (double)w.W4[k] * A0[j * HID + k];
    Y[j] = y;
  }
  if (want_grad) {
    // g3 = W4 .* d3  -> A1
    const double w4 = w.W4[j];
#pragma unroll
    for (int q = 0; q < MLP_R; ++q) A1[q * HID + j] = w4 * D3[q * HID + j];
    __syncthreads();
    // g2[k] = d2[k] * sum_j W3[j][k] g3[j]  -> A0 ;  g1[k] = d1[k] * sum_j W2[j][k] g2[j] -> A1
#pragma unroll 1
    for (int layer = 0; layer < 2; ++layer) {
      const float* W = layer == 0 ? w.W3 : w.W2;
      const double* Gin = layer == 0 ? A1 : A0;
      double* Gout = layer == 0 ? A0 : A1;
      const double* Dl = layer == 0 ? D2 : D1;
#pragma unroll
      for (int q = 0; q < MLP_R; ++q) acc[q] = 0.0;
#pragma unroll 4
      for (int k = 0; k < HID; ++k) {
        const double wv = W[k * HID + j];
#pragma unroll
        for (int q = 0; q < MLP_R; ++q) acc[q] += wv * Gin[q * HID + k];
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < MLP_R; ++q) Gout[q * HID + j] = acc[q] * Dl[q * HID + j];
      __syncthreads();
    }
    // gin[i] = sum_j W1[j][i] g1[j]
    if (j < MLP_R * NX) {
      const int q = j / NX, i = j % NX;
      double s = 0.0;
      for (int k = 0; k < HID; ++k) s += (double)w.W1[k * NX + i] * A1[q * HID + k];
      GIN[q * NX + i] = s;
    }
  }
  __syncthreads();
  if (j < MLP_R && valid[j]) {
    double grad[NX];
    const double c = nn_output(P, IN + j * NX, NRM[j], Y[j], want_grad ? GIN + j * NX : nullptr, want_grad ? grad : nullptr);
    double* o = (rows_mode == ROWS_FLAT) ? out11 + (size_t)rowb[j] * NN_OUT : out11 + ((size_t)rowb[j] * (N + 1) + rowk[j]) * NN_OUT;
    o[0] = c;
    if (want_grad)
#pragma unroll
      for (int q = 0; q < NX; ++q) o[1 + q] = grad[q];
  }
}

constexpr size_t MLP_SMEM = sizeof(double) * (5 * MLP_R * HID + MLP_R * NX * 2 + 2 * MLP_R);
// per device: called by smpc_create after cudaSetDevice
cudaError_t mlp_prepare() { return cudaFuncSetAttribute(mlp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MLP_SMEM); }

void launch_mlp(const LaunchCtx& c, const smpc_problem_t* dP, const MlpWeights& w, int B, int N, int rows_mode, int n_flat,
                const double* xsrc, const int32_t* r, const uint8_t* act, const uint8_t* need, double* out11, bool want_grad) {
  int n_rows = (rows_mode == ROWS_TERMINAL || rows_mode == ROWS_CAND) ? B : rows_mode == ROWS_ALL ? B * N : rows_mode == ROWS_RECEDING ? 2 * B : n_flat;
  if (rows_mode == ROWS_FLAT) B = n_flat;
  if (n_rows <= 0) return;
  const size_t smem = MLP_SMEM;
  mlp_kernel<<<GRID1D(n_rows, MLP_R), HID, smem, c.stream>>>(dP, w, B, N, rows_mode, n_rows, xsrc, r, act, need, out11, want_grad ? 1 : 0);
  ++*c.launches;
}

// ----------------------------------------------------------------------------------------------------------------
// Linearisation of every (problem, stage): one thread each (dev_model.cuh: linearize_stage)
// ----------------------------------------------------------------------------------------------------------------
#ifndef LIN_MINB
#define LIN_MINB 1
#endif
template <class R>
__global__ void __launch_bounds__(128, LIN_MINB)
linearize_kernel(const smpc_problem_t* __restrict__ dP, int B, int N, const double* __restrict__ xg, const double* __restrict__ ug,
                 const int32_t* __restrict__ r, const uint8_t* __restrict__ act, const double* __restrict__ nn11, const double* __restrict__ traj,
                 int n_traj, const int32_t* __restrict__ cur_step, R* lin) {
  // records are written tile-interleaved, [tile][stage][field][lane] (qp_split.cuh): thread = lane of warp (tile, stage),
  // so every field store of a warp is one contiguous 256-byte segment
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = idx & (TL - 1), w = idx / TL;
  const int tile = w / (N + 1), k = w % (N + 1);
  const int b = tile * TL + lane;
  if (b >= B) return;
  if (act && !act[b]) return;
  const smpc_problem_t& P = *dP;
  double x[NX], u[NU], xn[NX];
  const double* xb = xg + (size_t)b * (N + 1) * NX;
#pragma unroll
  for (int i = 0; i < NX; ++i) { x[i] = xb[k * NX + i]; xn[i] = (k < N) ? xb[(k + 1) * NX + i] : 0.0; }
#pragma unroll
  for (int i = 0; i < NU; ++i) u[i] = (k < N) ? ug[((size_t)b * N + k) * NU + i] : 0.0;
  const bool has_nn = stage_has_nn(P, k);
  bool gate = true;
  if (P.nn_rows == SMPC_NN_RECEDING && k < N) gate = (k == r[b]);      // controller.py:452-469
  if (P.nn_rows == SMPC_NN_PARALLEL) gate = (k == r[b]);               // controller.py:578-588 (r = candidate node of this solve)
  R* rec = lin + qs_blk(tile, N, k, REC, lane);
  const double* eer = n_traj > 0 ? traj + 3 * (size_t)min(cur_step[b] + k, n_traj - 1) : nullptr;     // controller.py:153-156
  linearize_stage(P, k, x, u, xn, has_nn, gate, nn11 + ((size_t)b * (N + 1) + k) * NN_OUT, rec, TL, eer);
}
// ----------------------------------------------------------------------------------------------------------------
// Linearisation, cooperative form: one CTA of eight warps per (tile of 32 problems, stage); lane = problem in every warp.
// The thread-per-stage form above keeps the state of the nominal passes (RNEA: 120 doubles, kinematics: 75) per thread and
// indexes it with run-time joint numbers: 255 registers, a 2 KB stack frame, 1.8 GB written per launch for 0.7 GB of records,
// FP64 pipe 36 % busy (profiles/r02_linearize_flops.md).  Here that state lives in shared memory, [field][lane], written once
// by the two nominal passes and read by everybody:
//   phase A   warp 0: recursive Newton-Euler pass (tau, body velocities / accelerations / wrenches)     warp 1: forward kinematics
//             warps 2-7: zero the record block (fields nobody writes must read 0)
//   phase B   the 15 columns of d tau / d(u, q, v) (one tangent recursion each), the 6 capsule pairs, the cost block and the
//             remaining rows are 23 independent items, dealt to the eight warps by estimated cost (longest first)
// Every item is the very function the thread-per-stage form calls (dev_model.cuh: lin_*), on the same operands.
// ----------------------------------------------------------------------------------------------------------------
constexpr int LC_WARPS = 8;
enum { LC_X = 0, LC_U = NX, LC_XN = NX + NU, LC_S = 2 * NX + NU, LC_K = LC_S + RS_SIZE, LC_FIELDS = LC_K + FK_SIZE };
constexpr size_t LC_SMEM = sizeof(double) * LC_FIELDS * TL;
// items: 0-4 d/du_j, 5-9 d/dq_j, 10-14 d/dv_j, 15-20 capsule pair, 21 cost block, 22 remaining rows; -1 = none
__constant__ int8_t lc_items[LC_WARPS][4] = {{5, 16, -1, -1}, {10, 17, -1, -1}, {6, 3, 9, -1}, {11, 15, 20, -1},
                                             {21, 2, 14, -1}, {7, 8, 18, -1},   {12, 13, 19, -1}, {0, 1, 4, 22}};

#ifndef LC_MINB
#define LC_MINB 2                // resident CTAs per SM the register allocation is sized for
#endif
template <class R>
__global__ void __launch_bounds__(32 * LC_WARPS, LC_MINB)
linearize_coop_kernel(const smpc_problem_t* __restrict__ dP, int B, int N, const double* __restrict__ xg, const double* __restrict__ ug,
                      const int32_t* __restrict__ r, const uint8_t* __restrict__ act, const double* __restrict__ nn11, const double* __restrict__ traj,
                      int n_traj, const int32_t* __restrict__ cur_step, R* lin) {
  extern __shared__ __align__(16) double lc_sm[];
  const smpc_problem_t& P = *dP;
  const int tile = blockIdx.x / (N + 1), k = blockIdx.x % (N + 1);
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int b = tile * TL + lane;
  const bool on = b < B && (!act || act[b]);
  if (!__any_sync(0xffffffffu, on)) return;                  // (the eight warps serve the same 32 problems: same answer)
  const bool term = (k == N);
  // guess of this stage (x, u) and state of the next one, staged once for all warps
  for (int e = threadIdx.x; e < LC_S * TL; e += 32 * LC_WARPS) {
    const int l = e & 31, f = e >> 5, bb = tile * TL + l;
    double v = 0.0;
    if (bb < B) {
      if (f < LC_U) v = xg[((size_t)bb * (N + 1) + k) * NX + f];
      else if (f < LC_XN) v = term ? 0.0 : ug[((size_t)bb * N + k) * NU + (f - LC_U)];
      else v = term ? 0.0 : xg[((size_t)bb * (N + 1) + k + 1) * NX + (f - LC_XN)];
    }
    lc_sm[e] = v;
  }
  __syncthreads();
  double x[NX], u[NU];
#pragma unroll
  for (int i = 0; i < NX; ++i) x[i] = lc_sm[(LC_X + i) * TL + lane];
#pragma unroll
  for (int i = 0; i < NU; ++i) u[i] = lc_sm[(LC_U + i) * TL + lane];
  RneaSm S{lc_sm + (size_t)LC_S * TL + lane};
  FkSm K{lc_sm + (size_t)LC_K * TL + lane};
  R* rec = lin + qs_blk(tile, N, k, REC, lane);
  double tau[NQ];
  if (wi == 0) {
    if (!term) rnea(P, P.inertial, x, x + NQ, u, S, tau);
  } else if (wi == 1) {
    fk(P, x, K);
  } else if (on) {
    for (int f = wi - 2; f < REC; f += LC_WARPS - 2) rec[(size_t)f * TL] = 0.0;
  }
  __syncthreads();
  if (!on) return;
  if (wi == 0 && !term) {
#pragma unroll
    for (int i = 0; i < NU; ++i) rec[(size_t)TL * (SMPC_REC_TAU + i)] = tau[i];
  }
  for (int s_ = 0; s_ < 4; ++s_) {
    const int item = lc_items[wi][s_];
    if (item < 0) break;
    if (item < 15) {
      if (term) continue;
      const int j = item % 5;
      if (item < 5) lin_tau_col<TAN_U>(P, S, x + NQ, u, j, rec, TL);
      else if (item < 10) lin_tau_col<TAN_Q>(P, S, x + NQ, u, j, rec, TL);
      else lin_tau_col<TAN_V>(P, S, x + NQ, u, j, rec, TL);
    } else if (item < 21) {
      if (k > 0 || P.stage0_collision_rows) lin_pair(P, K, item - 15, rec, TL);
    } else if (item == 21) {
      lin_cost(P, k, K, u, n_traj > 0 ? traj + 3 * (size_t)min(cur_step[b] + k, n_traj - 1) : P.ee_ref, rec, TL);
    } else {
      double xn[NX];
#pragma unroll
      for (int i = 0; i < NX; ++i) xn[i] = lc_sm[(LC_XN + i) * TL + lane];
      const bool has_nn = stage_has_nn(P, k);
      bool gate = true;
      if (P.nn_rows == SMPC_NN_RECEDING && k < N) gate = (k == r[b]);      // controller.py:452-469
      if (P.nn_rows == SMPC_NN_PARALLEL) gate = (k == r[b]);               // controller.py:578-588 (r = candidate node of this solve)
      lin_misc(P, k, x, u, xn, has_nn, gate, nn11 + ((size_t)b * (N + 1) + k) * NN_OUT, rec, TL);
    }
  }
}

// Which form runs: the thread-per-stage one.  The cooperative kernel gives the same bits but is slower on B200 (1.39 ms against 0.84 ms
// for 460 000 stages: its warps run eight different unrolled instruction streams and stall on instruction fetch and on the barrier
// behind the two nominal passes, profiles/r02_linearize.md); SMPC_LIN=coop selects it (read at every launch: a getenv per solve is noise).
static bool lin_thread_form() {
  const char* e = getenv("SMPC_LIN");
  return !(e && !strcmp(e, "coop"));
}
cudaError_t linearize_prepare() {
  cudaError_t e = cudaFuncSetAttribute(linearize_coop_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LC_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(linearize_coop_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LC_SMEM);
  return e;
}
void launch_linearize(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, const double* xg, const double* ug, const int32_t* r,
                      const uint8_t* act, const double* nn11, const double* traj, int n_traj, const int32_t* cur_step, void* lin, bool lin_f32) {
  const int tiles = (B + TL - 1) / TL;
  if (lin_thread_form()) {
    const int n = tiles * (N + 1) * TL;
    if (lin_f32) linearize_kernel<float><<<GRID1D(n, 128), 128, 0, c.stream>>>(dP, B, N, xg, ug, r, act, nn11, traj, n_traj, cur_step, static_cast<float*>(lin));
    else linearize_kernel<double><<<GRID1D(n, 128), 128, 0, c.stream>>>(dP, B, N, xg, ug, r, act, nn11, traj, n_traj, cur_step, static_cast<double*>(lin));
  } else {
    const int grid = tiles * (N + 1);
    if (lin_f32) linearize_coop_kernel<float><<<grid, 32 * LC_WARPS, LC_SMEM, c.stream>>>(dP, B, N, xg, ug, r, act, nn11, traj, n_traj, cur_step, static_cast<float*>(lin));
    else linearize_coop_kernel<double><<<grid, 32 * LC_WARPS, LC_SMEM, c.stream>>>(dP, B, N, xg, ug, r, act, nn11, traj, n_traj, cur_step, static_cast<double*>(lin));
  }
  ++*c.launches;
}

// ----------------------------------------------------------------------------------------------------------------
// Controller state machines after the solve (reference controller.py:274-284,311-315,375-388,477-498,541-565,651-660)
// ----------------------------------------------------------------------------------------------------------------
__device__ bool check_state_constraints_traj(const smpc_problem_t& P, const double* xt, int N) {
  // bounds on every row, collision on row 0 only (env_model.py:170-173 with the early return of :236-243)
  bool ok = true;
  for (int k = 0; k <= N; ++k) ok = ok && state_in_bounds(P, xt + k * NX);
  return ok && collision_free(P, xt);
}

__global__ void ctrl_post1_kernel(const smpc_problem_t* __restrict__ dP, int B, int N, const uint8_t* __restrict__ act,
                                  const double* __restrict__ xg, const double* __restrict__ ug, const double* __restrict__ xt,
                                  const int32_t* __restrict__ status, int32_t* fails, int32_t* r, double* x_viable, uint8_t* need_scan,
                                  uint8_t* abort_flag, double* u_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (act && !act[b]) return;
  const smpc_problem_t& P = *dP;
  const double* xgb = xg + (size_t)b * (N + 1) * NX;
  const double* ugb = ug + (size_t)b * N * NU;
  const double* xtb = xt + (size_t)b * (N + 1) * NX;
  const int st = status[b];
  need_scan[b] = 0;
  abort_flag[b] = 0;
  switch (P.controller) {
    case SMPC_CTRL_EVERYWHERE:
      if (st == 0 && check_state_constraints_traj(P, xtb, N)) fails[b] = 0; else fails[b] += 1;
      break;
    case SMPC_CTRL_STWA: case SMPC_CTRL_HTWA:
      if (st == 0 && check_state_constraints_traj(P, xtb, N)) fails[b] = 0;
      else {
        if (fails[b] == 0) for (int i = 0; i < NX; ++i) x_viable[(size_t)b * NX + i] = xgb[(N - 1) * NX + i];
        if (fails[b] == N - 1) { for (int i = 0; i < NU; ++i) u_out[(size_t)b * NU + i] = ugb[i]; abort_flag[b] = 1; }
        else fails[b] += 1;
      }
      break;
    case SMPC_CTRL_RECEDING: case SMPC_CTRL_REAL_RECEDING: {
      int rr = r[b];
      if (P.abort_flag) rr -= 1; else if (rr > 0) rr -= 1;
      if (rr == 0 && P.abort_flag) {
        for (int i = 0; i < NX; ++i) x_viable[(size_t)b * NX + i] = xgb[NX + i];
        rr = N;
        for (int i = 0; i < NU; ++i) u_out[(size_t)b * NU + i] = ugb[i];
        abort_flag[b] = 1;
      } else if (st == 0 && check_state_constraints_traj(P, xtb, N)) { fails[b] = 0; need_scan[b] = 1; }
      else fails[b] += 1;
      r[b] = rr;
      break;
    }
    default:   // naive, zerovel, st, backup
      if (st == 0) fails[b] = 0; else fails[b] += 1;
      break;
  }
}
void launch_ctrl_post1(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, const uint8_t* act, const double* xg, const double* ug,
                       const double* xt, int32_t* status, int32_t* fails, int32_t* r, double* x_viable, uint8_t* need_scan,
                       uint8_t* abort_flag, double* u_out) {
  ctrl_post1_kernel<<<GRID1D(B, 128), 128, 0, c.stream>>>(dP, B, N, act, xg, ug, xt, status, fails, r, x_viable, need_scan, abort_flag, u_out);
  ++*c.launches;
}

// receding-index update from the scan (controller.py:489-493) + provideControl (controller.py:169-184)
__global__ void ctrl_post2_kernel(const smpc_problem_t* __restrict__ dP, int B, int N, const uint8_t* __restrict__ act, double* xg, double* ug,
                                  const double* __restrict__ xt, const double* __restrict__ ut, const int32_t* __restrict__ fails, int32_t* r,
                                  int32_t* cur_step, const uint8_t* __restrict__ need_scan, const double* __restrict__ scan11,
                                  const uint8_t* __restrict__ abort_flag, double* u_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (act && !act[b]) return;
  if (abort_flag[b]) return;          // abort returns before the guess is shifted (controller.py:384-385,483-487)
  const smpc_problem_t& P = *dP;
  if (need_scan[b]) {
    int rr = r[b];
    for (int i = rr + 2; i <= N; ++i) {
      const double cval = scan11[((size_t)b * (N + 1) + i) * NN_OUT];
      if ((0.0 - P.tol_safe <= cval) && (cval <= 1e6 + P.tol_safe)) rr = i - 1;
    }
    r[b] = rr;
  }
  cur_step[b] += 1;
  double* xgb = xg + (size_t)b * (N + 1) * NX;
  double* ugb = ug + (size_t)b * N * NU;
  const double* xs = fails[b] > 0 ? xgb : xt + (size_t)b * (N + 1) * NX;
  const double* us = fails[b] > 0 ? ugb : ut + (size_t)b * N * NU;
  for (int i = 0; i < NU; ++i) u_out[(size_t)b * NU + i] = us[i];
  for (int i = 0; i < N * NX; ++i) xgb[i] = xs[NX + i];
  for (int i = 0; i < (N - 1) * NU; ++i) ugb[i] = us[NU + i];
  for (int i = 0; i < NX; ++i) xgb[N * NX + i] = xgb[(N - 1) * NX + i];
  for (int i = 0; i < NU; ++i) ugb[(N - 1) * NU + i] = ugb[(N - 2) * NU + i];
}
void launch_ctrl_post2(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, const uint8_t* act, double* xg, double* ug,
                       const double* xt, const double* ut, const int32_t* fails, int32_t* r, int32_t* cur_step, const uint8_t* need_scan,
                       const double* scan11, const uint8_t* abort_flag, double* u_out) {
  ctrl_post2_kernel<<<GRID1D(B, 128), 128, 0, c.stream>>>(dP, B, N, act, xg, ug, xt, ut, fails, r, cur_step, need_scan, scan11, abort_flag, u_out);
  ++*c.launches;
}

// ----------------------------------------------------------------------------------------------------------------
// ParallelController.step (controller.py:614-640): the host loops over the candidate nodes n = N .. 1 (one batched solve each);
// these kernels keep, per problem, the best node so far (sing_step :596-612) and finish the step.
// ----------------------------------------------------------------------------------------------------------------
__global__ void par_begin_kernel(int B, const uint8_t* __restrict__ act, int32_t* best, uint8_t* done, uint8_t* act2, int* n_open) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const bool on = !act || act[b];
  best[b] = 0; done[b] = 0; act2[b] = on ? 1 : 0;
  if (on) atomicAdd(n_open, 1);
}
void launch_par_begin(const LaunchCtx& c, int B, const uint8_t* act, int32_t* best, uint8_t* done, uint8_t* act2, int* n_open) {
  cudaMemsetAsync(n_open, 0, sizeof(int), c.stream);
  par_begin_kernel<<<GRID1D(B, 128), 128, 0, c.stream>>>(B, act, best, done, act2, n_open);
  ++*c.launches;
}

__global__ void par_eval_kernel(const smpc_problem_t* __restrict__ dP, int B, int N, int n, const uint8_t* __restrict__ act2_in,
                                const int32_t* __restrict__ status, const int32_t* __restrict__ r, const double* __restrict__ xt,
                                const double* __restrict__ ut, const double* __restrict__ scan11, int32_t* best, double* best_xt, double* best_ut,
                                uint8_t* done, uint8_t* act2_out, int* n_open) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B || !act2_in[b]) return;
  const smpc_problem_t& P = *dP;
  const double* xtb = xt + (size_t)b * (N + 1) * NX;
  const int rb = r[b];
  int checked_r = 0;                                               // check_safe_n (:590-595)
  for (int i = rb; i <= N; ++i) {
    const double cval = scan11[((size_t)b * (N + 1) + i) * NN_OUT];
    if (i >= 1 && (0.0 - P.tol_safe <= cval) && (cval <= 1e6 + P.tol_safe)) checked_r = i;
  }
  int result = 0;
  if (status[b] == 0) {
    const int constr_ver = checked_r >= rb ? checked_r : (n < rb ? n : rb);
    if (constr_ver - rb >= 0 && check_state_constraints_traj(P, xtb, N)) result = constr_ver;
  }
  if (result > best[b]) {
    best[b] = result;
    double* bx = best_xt + (size_t)b * (N + 1) * NX;
    double* bu = best_ut + (size_t)b * N * NU;
    const double* utb = ut + (size_t)b * N * NU;
    for (int i = 0; i < (N + 1) * NX; ++i) bx[i] = xtb[i];
    for (int i = 0; i < N * NU; ++i) bu[i] = utb[i];
    if (result == N) done[b] = 1;
  }
  const bool open = !done[b] && n > 1;
  act2_out[b] = open ? 1 : 0;
  if (open) atomicAdd(n_open, 1);
}
void launch_par_eval(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, int n, const uint8_t* act2_in, const int32_t* status, const int32_t* r,
                     const double* xt, const double* ut, const double* scan11, int32_t* best, double* best_xt, double* best_ut, uint8_t* done,
                     uint8_t* act2_out, int* n_open) {
  cudaMemsetAsync(n_open, 0, sizeof(int), c.stream);
  par_eval_kernel<<<GRID1D(B, 128), 128, 0, c.stream>>>(dP, B, N, n, act2_in, status, r, xt, ut, scan11, best, best_xt, best_ut, done, act2_out, n_open);
  ++*c.launches;
}

__global__ void par_post_kernel(const smpc_problem_t* __restrict__ dP, int B, int N, const uint8_t* __restrict__ act, const double* __restrict__ xg,
                                const double* __restrict__ ug, double* xt, double* ut, const int32_t* __restrict__ best,
                                const double* __restrict__ best_xt, const double* __restrict__ best_ut, int32_t* fails, int32_t* r, double* x_viable,
                                uint8_t* need_scan, uint8_t* abort_flag, double* u_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (act && !act[b]) return;
  need_scan[b] = 0;
  abort_flag[b] = 0;
  const double* xgb = xg + (size_t)b * (N + 1) * NX;
  const double* ugb = ug + (size_t)b * N * NU;
  if (best[b] > 1) {                                               // controller.py:625-629
    r[b] = best[b];
    double* xtb = xt + (size_t)b * (N + 1) * NX;
    double* utb = ut + (size_t)b * N * NU;
    const double* bx = best_xt + (size_t)b * (N + 1) * NX;
    const double* bu = best_ut + (size_t)b * N * NU;
    for (int i = 0; i < (N + 1) * NX; ++i) xtb[i] = bx[i];
    for (int i = 0; i < N * NU; ++i) utb[i] = bu[i];
    fails[b] = 0;
  } else {                                                         // :630-636
    fails[b] += 1;
    if (r[b] == 1) {
      for (int i = 0; i < NX; ++i) x_viable[(size_t)b * NX + i] = xgb[NX + i];
      r[b] = N;
      for (int i = 0; i < NU; ++i) u_out[(size_t)b * NU + i] = ugb[i];
      abort_flag[b] = 1;
      return;
    }
  }
  r[b] -= 1;                                                       // :637 (current_step and provideControl: ctrl_post2)
}
void launch_par_post(const LaunchCtx& c, const smpc_problem_t* dP, int B, int N, const uint8_t* act, const double* xg, const double* ug, double* xt,
                     double* ut, const int32_t* best, const double* best_xt, const double* best_ut, int32_t* fails, int32_t* r, double* x_viable,
                     uint8_t* need_scan, uint8_t* abort_flag, double* u_out) {
  par_post_kernel<<<GRID1D(B, 128), 128, 0, c.stream>>>(dP, B, N, act, xg, ug, xt, ut, best, best_xt, best_ut, fails, r, x_viable, need_scan, abort_flag, u_out);
  ++*c.launches;
}

// ----------------------------------------------------------------------------------------------------------------
// plant step, tau_fun, kinematics
// ----------------------------------------------------------------------------------------------------------------
__global__ void plant_kernel(const smpc_problem_t* __restrict__ dP, int B, const double* __restrict__ inertial, const double* __restrict__ noise,
                             const double* __restrict__ x, const double* __restrict__ u, const uint8_t* __restrict__ act, double* xn, double* a) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (act && !act[b]) return;
  double xx[NX], uu[NU], nn[NU], I[NQ][10], xo[NX], ao[NU];
  for (int i = 0; i < NX; ++i) xx[i] = x[(size_t)b * NX + i];
  for (int i = 0; i < NU; ++i) { uu[i] = u[(size_t)b * NU + i]; nn[i] = noise[(size_t)b * NU + i]; }
  for (int i = 0; i < NQ; ++i) for (int q = 0; q < 10; ++q) I[i][q] = inertial[((size_t)b * NQ + i) * 10 + q];
  plant_step(*dP, I, nn, xx, uu, xo, ao);
  for (int i = 0; i < NX; ++i) xn[(size_t)b * NX + i] = xo[i];
  if (a) for (int i = 0; i < NU; ++i) a[(size_t)b * NU + i] = ao[i];
}
void launch_plant(const LaunchCtx& c, const smpc_problem_t* dP, int B, const double* inertial, const double* noise, const double* x,
                  const double* u, const uint8_t* act, double* xn, double* a) {
  plant_kernel<<<GRID1D(B, 64), 64, 0, c.stream>>>(dP, B, inertial, noise, x, u, act, xn, a);
  ++*c.launches;
}

__global__ void tau_kernel(const smpc_problem_t* __restrict__ dP, int n, const double* __restrict__ x, const double* __restrict__ u, double* tau) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double xx[NX], uu[NU], t[NU];
  for (int q = 0; q < NX; ++q) xx[q] = x[(size_t)i * NX + q];
  for (int q = 0; q < NU; ++q) uu[q] = u[(size_t)i * NU + q];
  Rnea S;
  rnea(*dP, dP->inertial, xx, xx + NQ, uu, S, t);
  for (int q = 0; q < NU; ++q) tau[(size_t)i * NU + q] = t[q];
}
void launch_tau(const LaunchCtx& c, const smpc_problem_t* dP, int n, const double* x, const double* u, double* tau) {
  tau_kernel<<<GRID1D(n, 64), 64, 0, c.stream>>>(dP, n, x, u, tau);
  ++*c.launches;
}
// Torque-input dynamics, one explicit RK4 step with sensitivities (dev_model.cuh: rk4_sens; SURVEY.md section 8 row (f)4).  thread = row.
// The row's state / torque are read and its 160 outputs written with the caller's row-major layout: a warp's stores of one output
// field are strided by the row size, so the results are first collected in shared memory and written out by the whole CTA in
// consecutive addresses (one coalesced pass per output array).
constexpr int RK4_THREADS = 32;          // static shared memory: 32 x 101 doubles = 25.9 KB -> 8 CTAs (8 warps, the 255-register limit) per SM
template <bool SENS>
__global__ void __launch_bounds__(RK4_THREADS) rk4_sens_kernel(const smpc_problem_t* __restrict__ dP, int n, double dt, const double* __restrict__ x,
                                                              const double* __restrict__ tau, double* xn, double* A, double* B) {
  constexpr int LDS = NX * NX + 1;                            // A of one row + one padding word against bank conflicts
  __shared__ double so[SENS ? RK4_THREADS * LDS : 1];
  const int i0 = blockIdx.x * RK4_THREADS, i = i0 + threadIdx.x, rows = min(RK4_THREADS, n - i0);
  double xo[NX], Bo[SENS ? NX * NU : 1];
  if (i < n) {
    double xx[NX], tt[NU];
    for (int q = 0; q < NX; ++q) xx[q] = x[(size_t)i * NX + q];
    for (int q = 0; q < NU; ++q) tt[q] = tau[(size_t)i * NU + q];
    rk4_sens<SENS>(*dP, dP->inertial, dt, xx, tt, xo, SENS ? so + threadIdx.x * LDS : nullptr, Bo);
    for (int q = 0; q < NX; ++q) xn[(size_t)i * NX + q] = xo[q];
  }
  if (!SENS) return;
  __syncthreads();
  if (A) for (int e = threadIdx.x; e < rows * NX * NX; e += RK4_THREADS) A[(size_t)i0 * NX * NX + e] = so[(e / (NX * NX)) * LDS + e % (NX * NX)];
  if (B) {
    __syncthreads();
    if (i < n) for (int q = 0; q < NX * NU; ++q) so[threadIdx.x * LDS + q] = Bo[q];
    __syncthreads();
    for (int e = threadIdx.x; e < rows * NX * NU; e += RK4_THREADS) B[(size_t)i0 * NX * NU + e] = so[(e / (NX * NU)) * LDS + e % (NX * NU)];
  }
}
void launch_rk4_sens(const LaunchCtx& c, const smpc_problem_t* dP, int n, double dt, const double* x, const double* tau, double* xn, double* A, double* B) {
  if (A || B) rk4_sens_kernel<true><<<GRID1D(n, RK4_THREADS), RK4_THREADS, 0, c.stream>>>(dP, n, dt, x, tau, xn, A, B);
  else rk4_sens_kernel<false><<<GRID1D(n, RK4_THREADS), RK4_THREADS, 0, c.stream>>>(dP, n, dt, x, tau, xn, A, B);
  ++*c.launches;
}
__global__ void kin_kernel(const smpc_problem_t* __restrict__ dP, int n, const double* __restrict__ x, double* ee, double* dist) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double xx[NX], e[3], d[NPAIR];
  for (int q = 0; q < NX; ++q) xx[q] = x[(size_t)i * NX + q];
  distances(*dP, xx, e, d);
  if (ee) for (int q = 0; q < 3; ++q) ee[(size_t)i * 3 + q] = e[q];
  if (dist) for (int q = 0; q < NPAIR; ++q) dist[(size_t)i * NPAIR + q] = d[q];
}
void launch_kin(const LaunchCtx& c, const smpc_problem_t* dP, int n, const double* x, double* ee, double* dist) {
  kin_kernel<<<GRID1D(n, 64), 64, 0, c.stream>>>(dP, n, x, ee, dist);
  ++*c.launches;
}

__global__ void fill_i32_kernel(int32_t* p, int n, int32_t v) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }
void launch_fill_i32(const LaunchCtx& c, int32_t* p, int n, int32_t v) { fill_i32_kernel<<<GRID1D(n, 256), 256, 0, c.stream>>>(p, n, v); ++*c.launches; }
__global__ void fill_f64_kernel(double* p, size_t n, double v) { const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }
void launch_fill_f64(const LaunchCtx& c, double* p, size_t n, double v) { fill_f64_kernel<<<(unsigned)GRID1D(n, 256), 256, 0, c.stream>>>(p, n, v); ++*c.launches; }
__global__ void xv_from_guess_kernel(int B, int N, const double* xg, double* xv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * NX) return;
  const int b = i / NX, q = i % NX;
  xv[i] = xg[((size_t)b * (N + 1) + N) * NX + q];     // STWAController.setGuess (controller.py:390-393)
}
void launch_set_xviable_from_guess(const LaunchCtx& c, int B, int N, const double* xg, double* xv) {
  xv_from_guess_kernel<<<GRID1D(B * NX, 256), 256, 0, c.stream>>>(B, N, xg, xv);
  ++*c.launches;
}

// ----------------------------------------------------------------------------------------------------------------
// Closed loop (reference scripts/mpc.py:125-264).  Per problem: mode 0 = MPC, 1 = following the abort trajectory /
// PD hold, 2 = terminated.
// ----------------------------------------------------------------------------------------------------------------
// j < 0: a step captured into a CUDA graph -- the step index comes from the device (SIM_STEP_NEXT, kept by sim_post) and the backup
// request count at the start of the step is noted for the conditional node that decides on the backup solve (sim_backup_cond_kernel)
__global__ void sim_pre_kernel(SimDev s, const smpc_problem_t* __restrict__ dP, int j) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < 0 && b == 0) { s.counters[SIM_STEP_CUR] = s.counters[SIM_STEP_NEXT]; s.counters[SIM_REQ_SEEN] = s.counters[4]; }
  if (b >= s.B) return;
  const int Nb = s.Nb;
  s.need_ctrl[b] = 0; s.need_backup[b] = 0; s.live[b] = 0;
  if (s.mode[b] == 2) return;
  s.live[b] = 1;
  const double kp = 1.0, kd = 1e2;
  const double* x = s.x + (size_t)b * NX;
  if (s.mode[b] == 1) {                       // mpc.py:130-146
    const int ja = s.ja[b];
    const double* xa = s.x_abort + (size_t)b * (Nb + 1) * NX;
    const double* ua = s.u_abort + (size_t)b * Nb * NU;
    if (ja < Nb) {
      for (int i = 0; i < NQ; ++i) s.u[(size_t)b * NU + i] = ua[ja * NU + i] - (kp * (x[i] - xa[ja * NX + i]) + kd * (x[NQ + i] - xa[ja * NX + NQ + i]));
    } else {
      bool slow = true;
      for (int i = 0; i < NQ; ++i) slow = slow && (x[NQ + i] < 5e-3);          // no abs(), as upstream (mpc.py:138)
      if (slow) s.need_ctrl[b] = 1;
      else for (int i = 0; i < NQ; ++i) s.u[(size_t)b * NU + i] = -(kp * (x[i] - xa[Nb * NX + i]) + 3e2 * (x[NQ + i] - xa[Nb * NX + NQ + i]));
    }
    s.ja[b] = ja + 1;
  } else {
    s.need_ctrl[b] = 1;
  }
}
void launch_sim_pre(const LaunchCtx& c, const SimDev& s, const smpc_problem_t* dP, int j) {
  sim_pre_kernel<<<GRID1D(s.B, 128), 128, 0, c.stream>>>(s, dP, j);
  ++*c.launches;
}

// after controller.step: take its control; on a fresh abort prepare the backup OCP (mpc.py:161-177)
__global__ void sim_mid_kernel(SimDev s, const double* __restrict__ x_viable, double* bk_xg, double* bk_ug, const int32_t* __restrict__ qp_iter_main) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= s.B) return;
  if (!s.need_ctrl[b]) return;
  const int Nb = s.Nb;
  for (int i = 0; i < NU; ++i) s.u[(size_t)b * NU + i] = s.u_ctrl[(size_t)b * NU + i];
  atomicAdd(&s.counters[0], 1ull);
  atomicAdd(&s.counters[3], (unsigned long long)qp_iter_main[b]);
  const bool sa = s.abort_flag[b] != 0;
  if (s.mode[b] == 1) {          // came back from an abort: a repeated abort does NOT re-solve the backup (mpc.py:138-141)
    s.mode[b] = sa ? 1 : 0;
    return;
  }
  if (sa) {
    const double* xv = x_viable + (size_t)b * NX;
    if (!(s.outcome[b] & SMPC_OUT_ABORTED)) for (int i = 0; i < NX; ++i) s.xv_first[(size_t)b * NX + i] = xv[i];
    double* xg = bk_xg + (size_t)b * (Nb + 1) * NX;
    double* ug = bk_ug + (size_t)b * Nb * NU;
    for (int k = 0; k <= Nb; ++k) for (int i = 0; i < NX; ++i) xg[k * NX + i] = xv[i];
    for (int i = 0; i < Nb * NU; ++i) ug[i] = 0.0;
    s.need_backup[b] = 1;
    atomicAdd(&s.counters[4], 1ull);
  }
}
void launch_sim_mid(const LaunchCtx& c, const SimDev& s, const double* x_viable, double* bk_xg, double* bk_ug, const int32_t* qp_iter_main) {
  sim_mid_kernel<<<GRID1D(s.B, 128), 128, 0, c.stream>>>(s, x_viable, bk_xg, bk_ug, qp_iter_main);
  ++*c.launches;
}

// backup result, plant step, bounds / collision checks, logging (mpc.py:178-190,240-264)
__global__ void sim_post_kernel(SimDev s, const smpc_problem_t* __restrict__ dP, int j, const int32_t* __restrict__ bk_status,
                                const double* __restrict__ bk_xt, const double* __restrict__ bk_ut, const double* __restrict__ inertial,
                                const double* __restrict__ noise, const int32_t* __restrict__ qp_iter_bk) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < 0) j = (int)s.counters[SIM_STEP_CUR];
  if (b == 0) s.counters[SIM_STEP_NEXT] = (unsigned long long)j + 1;
  if (b >= s.B || j >= s.n_steps) return;          // (a replay past the end of the log does nothing)
  if (!s.live[b]) return;
  const smpc_problem_t& P = *dP;
  const int Nb = s.Nb;
  bool done = false;
  if (s.need_backup[b]) {
    atomicAdd(&s.counters[1], 1ull);
    atomicAdd(&s.counters[3], (unsigned long long)qp_iter_bk[b]);
    if (bk_status[b] != 0) { s.outcome[b] |= SMPC_OUT_COLLIDED; done = true; }
    else {
      s.ja[b] = 0;
      s.outcome[b] |= SMPC_OUT_ABORTED;
      s.mode[b] = 1;
      for (int i = 0; i < (Nb + 1) * NX; ++i) s.x_abort[(size_t)b * (Nb + 1) * NX + i] = bk_xt[(size_t)b * (Nb + 1) * NX + i];
      for (int i = 0; i < Nb * NU; ++i) s.u_abort[(size_t)b * Nb * NU + i] = bk_ut[(size_t)b * Nb * NU + i];
    }
  }
  double xx[NX], uu[NU], nn[NU], I[NQ][10], xo[NX], ao[NU];
  for (int i = 0; i < NU; ++i) { uu[i] = s.u[(size_t)b * NU + i]; s.ulog[((size_t)b * s.n_steps + j) * NU + i] = uu[i]; }
  if (done) { s.mode[b] = 2; return; }
  for (int i = 0; i < NX; ++i) xx[i] = s.x[(size_t)b * NX + i];
  for (int i = 0; i < NU; ++i) nn[i] = noise[(size_t)b * NU + i];
  for (int i = 0; i < NQ; ++i) for (int q = 0; q < 10; ++q) I[i][q] = inertial[((size_t)b * NQ + i) * 10 + q];
  plant_step(P, I, nn, xx, uu, xo, ao);
  atomicAdd(&s.counters[2], 1ull);
  for (int i = 0; i < NX; ++i) { s.xlog[((size_t)b * (s.n_steps + 1) + j + 1) * NX + i] = xo[i]; s.x[(size_t)b * NX + i] = xo[i]; }
  if (!state_in_bounds(P, xo) || !collision_free(P, xo)) { s.outcome[b] |= SMPC_OUT_COLLIDED; s.mode[b] = 2; }
}
void launch_sim_post(const LaunchCtx& c, const SimDev& s, const smpc_problem_t* dP, int j, const int32_t* bk_status, const double* bk_xt,
                     const double* bk_ut, const double* inertial, const double* noise, const int32_t* qp_iter_bk) {
  sim_post_kernel<<<GRID1D(s.B, 64), 64, 0, c.stream>>>(s, dP, j, bk_status, bk_xt, bk_ut, inertial, noise, qp_iter_bk);
  ++*c.launches;
}

// convergence test of mpc.py:273 on the last logged state (NaN after an early exit -> not converged)
__global__ void sim_outcome_kernel(SimDev s, const smpc_problem_t* __restrict__ dP, int32_t* out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= s.B) return;
  const smpc_problem_t& P = *dP;
  double xx[NX], ee[3];
  for (int i = 0; i < NX; ++i) xx[i] = s.xlog[((size_t)b * (s.n_steps + 1) + s.n_steps) * NX + i];
  distances(P, xx, ee, nullptr);
  double d2 = 0.0;
  for (int k = 0; k < 3; ++k) d2 += (ee[k] - P.ee_ref[k]) * (ee[k] - P.ee_ref[k]);
  int o = s.outcome[b] & ~SMPC_OUT_CONVERGED;
  if (sqrt(d2) < P.tol_conv) o |= SMPC_OUT_CONVERGED;
  out[b] = o;
}
// condition of the conditional IF node around the backup solve of a captured step: some problem asked for it in this step
__global__ void __launch_bounds__(1) sim_backup_cond_kernel(const unsigned long long* __restrict__ counters, cudaGraphConditionalHandle cond) {
  cudaGraphSetConditional(cond, counters[4] != counters[SIM_REQ_SEEN] ? 1u : 0u);
}
void launch_sim_backup_cond(const LaunchCtx& c, const SimDev& s, cudaGraphConditionalHandle cond) {
  sim_backup_cond_kernel<<<1, 1, 0, c.stream>>>(s.counters, cond);
  ++*c.launches;
}

void launch_sim_outcome(const LaunchCtx& c, const SimDev& s, const smpc_problem_t* dP, int32_t* out) {
  sim_outcome_kernel<<<GRID1D(s.B, 128), 128, 0, c.stream>>>(s, dP, out);
  ++*c.launches;
}

}  // namespace smpc
