// QP kernels: the phases of the split interior-point solver of qp_split.cuh, one small kernel each, and the host loop
// that sequences them.  Replaces the HPIPM solve inside AcadosOcpSolver.solve() (reference controller.py:158) and the
// full-step update / status mapping that acados' SQP_RTI performs around it (controller.py:161-167).
//
// Launch shapes (B problems, T = ceil(B/32) tiles, N+1 stages):
//   prep / step   one warp per (tile, stage): T (N+1) warps, 4 warps per CTA; lane = problem of the tile.  Streaming
//                 kernels: every global access of a warp is one contiguous 256-byte segment of the tile-interleaved arrays.
//   ric1 / ric2   one warp per tile (lane = problem), walking the stages; ric1 keeps P_{k+1}, p_{k+1} of its 32 problems
//                 in shared memory (33 KB per warp).
//   ctl / red     one thread per problem.
// The host reads two counters (problems still active, problems that asked for the centering re-solve) once per IPM
// iteration; everything else is asynchronous on the handle's stream.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "engine.cuh"

namespace smpc {
inline namespace QS_FLAVOUR {

namespace {

#ifndef QS_SP_WARPS
#define QS_SP_WARPS 2            // (2 / 4 / 8 warps per CTA at the same 8 warps per SM: cfg[1] 53.2 / 53.5 / 54.0 ms per step, gpurun_out/r2c46)
#endif
constexpr int SP_WARPS = QS_SP_WARPS;   // warps per CTA of the stage-parallel kernels
#ifndef QS_RIC_NBUF
#define QS_RIC_NBUF 1            // staging buffers of the Riccati sweeps (1: more resident warps per SM, no fetch overlap)
#endif
#ifndef QS_PREP_MINB
#define QS_PREP_MINB 4
#endif
#ifndef QS_PC_SBND
#define QS_PC_SBND 1             // cooperative prep: row bounds of the stage in shared memory (prep 13.6 -> 13.0 ms per cfg[1] solve, gpurun_out/r2c34)
#endif
#ifndef QS_PC_ROLL
#define QS_PC_ROLL 1             // unroll factor of the row loops of the cooperative prep kernel (1 = rolled)
#endif
constexpr int PC_ROLL = QS_PC_ROLL;
#ifndef QS_SP_MINB
#define QS_SP_MINB 4             // resident CTAs (of SP_WARPS = 2 warps) per SM the register allocation of the step kernels is sized for: 255 registers, no spills, 8 warps
                                 // per SM.  Measured with four warps per CTA and one tile group (gpurun_out/r2c43): 8 warps per SM 53.4 ms per cfg[1] step, 12 warps
                                 // (168 registers, spills between the load phases: the round-1 setting, found with three concurrent tile groups) 55.0 ms, 16 warps 59.9 ms
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__global__ void __launch_bounds__(32) qs_init_kernel(QsBufs q, int B, const double* __restrict__ x0, const int32_t* __restrict__ r,
                                                      const uint8_t* __restrict__ act) {
  qs_init(q, blockIdx.x, threadIdx.x, B, x0, r, act);
}

constexpr size_t PREP_SMEM = sizeof(double) * 2 * PREP_SCRATCH * TL + 512;   // a retiring prep CTA leaves room for one Riccati CTA
constexpr int PREP_WARPS = 2;    // warps per CTA of prep: 2 x 26.9 KB of lane-private Jacobian scratch, 4 CTAs per SM
template <bool FIRST>
__global__ void __launch_bounds__(32 * PREP_WARPS, QS_PREP_MINB) qs_prep_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int T, int kk,
                                                                                          const int* __restrict__ kk_dev) {
  if (kk_dev) kk = *kk_dev;
  extern __shared__ __align__(128) double jsm_all[];
  const int wi = threadIdx.x >> 5;
  const int w = blockIdx.x * PREP_WARPS + wi;
  if (w >= T * (q.N + 1)) return;
  qs_prep<FIRST>(*dP, q, w / (q.N + 1), threadIdx.x & 31, w % (q.N + 1), kk, jsm_all + (size_t)wi * PREP_SCRATCH * TL + (threadIdx.x & 31));
}

// ---------------------------------------------------------------------------------------------------------------
// prep, cooperative form (IPM iterations kk >= 1): one CTA of four warps per (tile, stage).
// The whole input of the work item -- stage record, previous iterate, step: 107.5 KB -- is staged into shared memory by three
// TMA bulk copies, so no warp ever waits on a global load in the middle of its instruction stream (the thread-per-stage form
// above spends 14 of 23 cycles per instruction there, profiles/r01_qp_v6_launches.md); the instruction stream of qs_prep is
// split over the four warps (lane = problem in all of them):
//   rows    warp 0: iterate update, stationarity base, dynamics residual, box rows 0-3     warp 1: box rows 4-9
//           warp 2: torque rows                                                           warp 3: capsule rows + viability row
//           every row leaves (nu = lam_u - lam_l, gam = c_l - c_u, G = G_l + G_u) in the shared-memory slots of its own,
//           already consumed, multipliers; every warp leaves its residual-norm partials the same way
//   merge   warp 0: C' nu, C' gam -> stationarity residual and affine gradient, norms     warps 1-3: rows of H + C' G C
// Same arithmetic per term and the same summation orders as qs_prep<false>: the two forms agree to the last bit.
// ---------------------------------------------------------------------------------------------------------------
constexpr int PC_REC0 = SMPC_REC_X;                       // first staged record field (the controls of the guess are not needed)
constexpr int PC_NREC = 180;                              // staged record fields [5, 185)
constexpr int PC_WARPS = 4;
constexpr int PC_NPART = 6;                               // residual-norm partials per warp
// staged: previous iterate (fp64), stage record and step (storage type); the fp32 flavour keeps the fp64 partials of the warps in an array of
// their own (the fp64 flavour parks them in consumed slots of the staged step, as before: two CTAs of 107.5 KB per SM)
constexpr size_t PC_SMEM = sizeof(double) * NIT * TL + sizeof(qs_real) * (PC_NREC + NIT) * TL +
                           (sizeof(qs_real) == 8 ? 0 : sizeof(double) * PC_WARPS * PC_NPART * TL) + 16 + sizeof(double) * 36;
static_assert(PC_REC0 + PC_NREC > SMPC_REC_HQ && PC_REC0 + PC_NREC <= SMPC_REC, "staged record range");

__device__ __forceinline__ void pc_row_out(double* s_it, int sl, double nu, double gam, double G) {
  QF(s_it, I_LAM + sl) = nu; QF(s_it, I_LAM + QNR + sl) = gam; QF(s_it, I_T + sl) = G;
}

__global__ void __launch_bounds__(32 * PC_WARPS, 2) qs_prep_coop_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int T, int kk,
                                                                      const int* __restrict__ kk_dev) {
  if (kk_dev) kk = *kk_dev;
  extern __shared__ __align__(128) double pc_sm[];
  const smpc_problem_t& P = *dP;
  const int N = q.N;
  const int tile = blockIdx.x / (N + 1), k = blockIdx.x % (N + 1);
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  const bool on = QF(pi, J_ACT) != 0;
  if (!__any_sync(0xffffffffu, on)) return;               // (same decision in the four warps: same tile)
  const qs_real* g_rec_blk = q.rec + qs_blk(tile, N, k, REC, 0);
  const double* g_it_blk = q.it[(kk & 1) ^ 1] + qs_blk(tile, N, k, NIT, 0);
  const qs_real* g_st_blk = q.st + qs_blk(tile, N, k, NIT, 0);
  double* sm_it = pc_sm;
  qs_real* sm_rec = reinterpret_cast<qs_real*>(sm_it + (size_t)NIT * TL);
  qs_real* sm_st = sm_rec + (size_t)PC_NREC * TL;
  double* sm_part = reinterpret_cast<double*>(sm_st + (size_t)NIT * TL);           // fp32 flavour only
  uint64_t* bar = reinterpret_cast<uint64_t*>(sm_part + (sizeof(qs_real) == 8 ? 0 : (size_t)PC_WARPS * PC_NPART * TL));
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const uint32_t nb_rec = PC_NREC * TL * sizeof(qs_real), nb_it = NIT * TL * 8, nb_st = NIT * TL * sizeof(qs_real);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(nb_rec + nb_it + nb_st) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sm_rec)),
                 "l"(g_rec_blk + (size_t)PC_REC0 * TL), "r"(nb_rec), "r"(smem_u32(bar)) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sm_it)),
                 "l"(g_it_blk), "r"(nb_it), "r"(smem_u32(bar)) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sm_st)),
                 "l"(g_st_blk), "r"(nb_st), "r"(smem_u32(bar)) : "memory");
  }
  // (tried: issuing the staging before the activity flags are read, so that the two round trips overlap -- 0.3 ms per step slower)
  const StageFlags F = qs_flags(P, k);
  // bounds of the rows of this stage -> shared memory: the row loops are rolled, and a bound read from the problem block in global memory
  // with a run-time row index would put a load round trip into every iteration (ncu source page: 6.6 % of the samples on those DADDs)
  double* sbnd = reinterpret_cast<double*>(bar + 2);        // [0,10) box lower, [10,20) box upper, [20,25) [25,30) torque, [30,36) capsule lower
  if (QS_PC_SBND && threadIdx.x < 36) {
    const int t = threadIdx.x;
    const bool rr = P.controller == SMPC_CTRL_REAL_RECEDING;
    double v;
    if (t < 10) v = k == N ? P.lbx_e[t] : (rr ? P.x_min[t] : P.lbx[t]);
    else if (t < 20) v = k == N ? P.ubx_e[t - 10] : (rr ? P.x_max[t - 10] : P.ubx[t - 10]);
    else if (t < 25) v = P.tau_min[t - 20];
    else if (t < 30) v = P.tau_max[t - 25];
    else v = P.pair_lo_ocp[t - 30];
    sbnd[t] = v;
  }
  // lane views: field f of the record at rs[f * TL] (valid for PC_REC0 <= f < PC_REC0 + PC_NREC)
  const qs_real* rs = sm_rec - (size_t)PC_REC0 * TL + lane;
  double* s_it = sm_it + lane;
  const qs_real* s_st = sm_st + lane;
  // partial j of warp w: fp64 flavour -> the consumed step slots of the warp's first rows (warp 0: box 0-2; 1: box 4-6; 2: torque 0-2;
  // 3: capsule 0-2), fp32 flavour -> sm_part
  auto part = [&](int w, int j) -> double& {
    if (sizeof(qs_real) == 8) {
      const int s0 = w == 0 ? 0 : (w == 1 ? 4 : (w == 2 ? 10 : 15));
      const int slot = (j & 1) ? I_LAM + QNR + s0 + (j >> 1) : I_LAM + s0 + (j >> 1);
      return *reinterpret_cast<double*>(const_cast<qs_real*>(s_st) + (size_t)slot * TL);
    }
    return sm_part[(size_t)(w * PC_NPART + j) * TL + lane];
  };
  const double* pd = q.pd + qs_pb(tile, NPD, lane);
  const double a = QF(pd, D_STEP);
  const int rrec = QF(pi, J_R);
  double* ito = q.it[kk & 1] + qs_blk(tile, N, k, NIT, lane);
  qs_real* hc = q.sb + qs_blk(tile, N, k, NHC, lane);
  const double lam_min = 1e-16, t_min = 1e-16, reg = P.qp_reg_prim;
  const double dt = P.dt, a2 = 0.5 * P.dt * P.dt;

  // neighbour data of warp 0 (global; issued before the wait so that the round trip overlaps the staging)
  double pqn[10], znx[10];
  if (wi == 0) {
#pragma unroll
    for (int j = 0; j < 10; ++j) { pqn[j] = 0.0; znx[j] = 0.0; }
    if (k < N) {
      const double* itn = q.it[(kk & 1) ^ 1] + qs_blk(tile, N, k + 1, NIT, lane);
      const qs_real* stn = q.st + qs_blk(tile, N, k + 1, NIT, lane);
#pragma unroll
      for (int j = 0; j < 10; ++j) {
        pqn[j] = QF(itn, I_PIM + j) + a * QF(stn, I_PIM + j);
        znx[j] = QF(itn, I_Z + 5 + j) + a * QF(stn, I_Z + 5 + j);
      }
    }
  }
  __syncthreads();                                         // barrier initialised before anyone polls it
  {
    uint32_t ok;
    do {
      asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(smem_u32(bar)), "r"(0) : "memory");
    } while (!ok);
  }

  // ---- iterate of this stage (every warp) ----
  double z[15];
#pragma unroll
  for (int i = 0; i < 15; ++i) z[i] = QF(s_it, I_Z + i) + a * QF(s_st, I_Z + i);
  if (k == N) {
#pragma unroll
    for (int i = 0; i < 5; ++i) z[i] = 0.0;
  }
  // box of dx_j (qs_box with the record of this stage in shared memory)
  auto box = [&](int j, double& lo, double& hi) {
    const double xk = QF(rs, SMPC_REC_X + j);
    if (k == 0) { lo = QF(pd, D_X0 + j) - xk; hi = lo; }
    else if (k < N && P.controller == SMPC_CTRL_REAL_RECEDING && k == rrec) {
      const double c = QF(q.rec + qs_blk(tile, N, k + 1, REC, lane), SMPC_REC_X + j); lo = c - 1e-3 - xk; hi = c + 1e-3 - xk;
    }
#if QS_PC_SBND
    else { lo = sbnd[j] - xk; hi = sbnd[10 + j] - xk; }
#else
    else if (k == N) { lo = P.lbx_e[j] - xk; hi = P.ubx_e[j] - xk; }
    else if (P.controller == SMPC_CTRL_REAL_RECEDING) { lo = P.x_min[j] - xk; hi = P.x_max[j] - xk; }
    else { lo = P.lbx[j] - xk; hi = P.ubx[j] - xk; }
#endif
  };
  QsNorms nr;
  nr.ng = nr.nb = nr.nd = nr.nm = nr.mu = nr.chk = 0.0; nr.cnt = 0;
  auto upd = [&](int slot, double& lam, double& t) {
    lam = fmax(QF(s_it, I_LAM + slot) + a * QF(s_st, I_LAM + slot), lam_min);
    t = fmax(QF(s_it, I_T + slot) + a * QF(s_st, I_T + slot), t_min);
  };
  auto side = [&](int slot, double sgn, double az, double bnd, double slack, double lam, double t, double& G, double& c) {
    if (on) { QF(ito, I_LAM + slot) = lam; QF(ito, I_T + slot) = t; }
    const double r = t - (sgn * (az - bnd) + slack);
    const double rm = QS_MUL(lam, t);                      // (QS_MUL: see the note at its definition)
    const double it_ = QS_SRCP(t);
    G = QS_MUL(lam, it_);
    c = QS_MUL(fma(-lam, r, rm), it_);
    nr.mu += rm; nr.chk += rm + r; nr.nm = fmax(nr.nm, fabs(rm)); nr.nd = fmax(nr.nd, fabs(r)); nr.cnt += 1;
  };
  // a hard two-sided row: update, residuals, (nu, gam, G) into the row's own shared-memory slots
  auto hard_row = [&](int sl, double az, double lo, double hi) {
    double ll, tl, lu, tu, Gl, Gu, cl, cu;
    upd(sl, ll, tl); upd(QNR + sl, lu, tu);
    side(sl, 1.0, az, lo, 0.0, ll, tl, Gl, cl);
    side(QNR + sl, -1.0, az, hi, 0.0, lu, tu, Gu, cu);
    pc_row_out(s_it, sl, lu - ll, cl - cu, Gl + Gu);
  };

  double rg[15];                                           // warp 0: stationarity residual without the inequality multipliers
  if (wi == 0) {
    const double hu = QF(rs, SMPC_REC_HU), hq = QF(rs, SMPC_REC_HQ), hv = QF(rs, SMPC_REC_HV);
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      rg[i] = (k == N) ? 0.0 : hu * z[i] + QF(rs, SMPC_REC_G + i);
      double s = QF(rs, SMPC_REC_G + 5 + i) + hq * z[5 + i];
#pragma unroll
      for (int j = 0; j < 5; ++j) s += QF(rs, SMPC_REC_HQQ + trs(i, j)) * z[5 + j];
      rg[5 + i] = s;
      rg[10 + i] = QF(rs, SMPC_REC_G + 10 + i) + hv * z[10 + i];
    }
    double pimv[10];
#pragma unroll
    for (int j = 0; j < 10; ++j) {
      pimv[j] = (k == 0) ? 0.0 : QF(s_it, I_PIM + j) + a * QF(s_st, I_PIM + j);
      rg[5 + j] -= pimv[j];
    }
    if (k < N) {
      double rb[10];
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        rb[j] = z[5 + j] + dt * z[10 + j] + a2 * z[j] + QF(rs, SMPC_REC_B + j);
        rb[5 + j] = z[10 + j] + dt * z[j] + QF(rs, SMPC_REC_B + 5 + j);
        const double pq = pqn[j], pv = pqn[5 + j];
        rg[j] += fma(a2, pq, QS_MUL(dt, pv));
        rg[5 + j] += pq;
        rg[10 + j] += dt * pq + pv;
        rb[j] -= znx[j];
        rb[5 + j] -= znx[5 + j];
      }
#pragma unroll
      for (int j = 0; j < 10; ++j) { if (on) QF(hc, H_RB + j) = rb[j]; nr.nb = fmax(nr.nb, fabs(rb[j])); nr.chk += rb[j]; }
    }
    if (on) {
#pragma unroll
      for (int i = 0; i < 15; ++i) QF(ito, I_Z + i) = z[i];
#pragma unroll
      for (int j = 0; j < 10; ++j) QF(ito, I_PIM + j) = pimv[j];
    }
    // (row loops are ROLLED, QS_PC_ROLL: the kernel is 111 KB of straight-line SASS run once per CTA by four warps at four different program
    // counters, and the instruction fetch was its largest stall -- ncu: no_instruction 3.7 of 11 cycles per issue, L1.5 I-cache 32 KB)
#pragma unroll PC_ROLL
    for (int j = 0; j < 4; ++j) { double lo, hi; box(j, lo, hi); hard_row(j, QF(s_it, I_Z + 5 + j) + a * QF(s_st, I_Z + 5 + j), lo, hi); }
  } else if (wi == 1) {
#pragma unroll PC_ROLL
    for (int j = 4; j < 10; ++j) { double lo, hi; box(j, lo, hi); hard_row(j, QF(s_it, I_Z + 5 + j) + a * QF(s_st, I_Z + 5 + j), lo, hi); }
  } else if (wi == 2) {
    if (F.tau) {
#pragma unroll PC_ROLL
      for (int r = 0; r < 5; ++r) {
        double az = 0.0;
#pragma unroll
        for (int c = 0; c < 15; ++c) az += QF(rs, SMPC_REC_JTAU + r * 15 + c) * z[c];
        const double v = QF(rs, SMPC_REC_TAU + r);
#if QS_PC_SBND
        hard_row(10 + r, az, sbnd[20 + r] - v, sbnd[25 + r] - v);
#else
        hard_row(10 + r, az, P.tau_min[r] - v, P.tau_max[r] - v);
#endif
      }
    }
  } else {
    if (F.dist) {
#pragma unroll PC_ROLL
      for (int p = 0; p < 6; ++p) {
        double az = 0.0;
#pragma unroll
        for (int c = 0; c < 5; ++c) az += QF(rs, SMPC_REC_JDIST + p * 5 + c) * z[5 + c];
        const double v = QF(rs, SMPC_REC_DIST + p);
#if QS_PC_SBND
        hard_row(15 + p, az, sbnd[30 + p] - v, P.pair_hi - v);
#else
        hard_row(15 + p, az, P.pair_lo_ocp[p] - v, P.pair_hi - v);
#endif
      }
    }
    if (F.nn) {
      double az = 0.0;
#pragma unroll
      for (int c = 0; c < 10; ++c) az += QF(rs, SMPC_REC_JNN + c) * z[5 + c];
      const double v = QF(rs, SMPC_REC_NN);
      double sl[2] = {0.0, 0.0}, ls[2] = {0.0, 0.0}, ts[2] = {0.0, 0.0};
      if (F.soft) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          sl[h] = QF(s_it, I_SLK + h) + a * QF(s_st, I_SLK + h);
          ls[h] = fmax(QF(s_it, I_SLK + 2 + h) + a * QF(s_st, I_SLK + 2 + h), lam_min);
          ts[h] = fmax(QF(s_it, I_SLK + 4 + h) + a * QF(s_st, I_SLK + 4 + h), t_min);
        }
      }
      if (on) {
#pragma unroll
        for (int h = 0; h < 2; ++h) { QF(ito, I_SLK + h) = sl[h]; QF(ito, I_SLK + 2 + h) = ls[h]; QF(ito, I_SLK + 4 + h) = ts[h]; }
      }
      double ll, tl, lu, tu, Gl, Gu, cl, cu;
      upd(21, ll, tl); upd(QNR + 21, lu, tu);
      side(21, 1.0, az, 0.0 - v, sl[0], ll, tl, Gl, cl);
      side(QNR + 21, -1.0, az, 1e6 - v, sl[1], lu, tu, Gu, cu);
      if (F.soft) {
        const double lam2[2] = {ll, lu};
        double G2[2] = {Gl, Gu}, c2[2] = {cl, cu};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const double rsl = ts[h] - sl[h];
          const double rgs = F.zpen - lam2[h] - ls[h];
          const double rms = QS_MUL(ls[h], ts[h]);
          const double its = QS_SRCP(ts[h]);
          const double Gs = QS_MUL(ls[h], its);
          const double cs = QS_MUL(fma(-ls[h], rsl, rms), its);
          const double Wl = QS_SRCP(G2[h] + Gs);
          c2[h] = c2[h] - G2[h] * Wl * (rgs + c2[h] + cs);
          G2[h] = G2[h] * Gs * Wl;
          nr.mu += rms; nr.chk += rms + rsl + rgs;
          nr.nm = fmax(nr.nm, fabs(rms)); nr.nd = fmax(nr.nd, fabs(rsl)); nr.ng = fmax(nr.ng, fabs(rgs));
          nr.cnt += 1;
        }
        Gl = G2[0]; Gu = G2[1]; cl = c2[0]; cu = c2[1];
      }
      pc_row_out(s_it, 21, lu - ll, cl - cu, Gl + Gu);
    }
  }
  // residual-norm partials of this warp -> consumed step slots of its first rows (warp 0: box 0-2; 1: box 4-6; 2: torque 0-2; 3: capsule 0-2)
  {
    part(wi, 0) = nr.chk; part(wi, 1) = nr.nm; part(wi, 2) = nr.nd;
    part(wi, 3) = nr.ng; part(wi, 4) = (double)nr.cnt;
    part(wi, 5) = nr.mu;
  }
  __syncthreads();

  if (wi == 0) {
    // ---- merge: rg += C' nu, gd = C' gam; norms; affine gradient ----
    double gd[15];
#pragma unroll
    for (int i = 0; i < 15; ++i) gd[i] = 0.0;
#pragma unroll
    for (int j = 0; j < 10; ++j) { rg[5 + j] += QF(s_it, I_LAM + j); gd[5 + j] += QF(s_it, I_LAM + QNR + j); }
    if (F.tau) {
#pragma unroll PC_ROLL
      for (int r = 0; r < 5; ++r) {
        const double nu = QF(s_it, I_LAM + 10 + r), gam = QF(s_it, I_LAM + QNR + 10 + r);
#pragma unroll
        for (int c = 0; c < 15; ++c) { const double jv = QF(rs, SMPC_REC_JTAU + r * 15 + c); rg[c] += jv * nu; gd[c] += jv * gam; }
      }
    }
    if (F.dist) {
#pragma unroll PC_ROLL
      for (int p = 0; p < 6; ++p) {
        const double nu = QF(s_it, I_LAM + 15 + p), gam = QF(s_it, I_LAM + QNR + 15 + p);
#pragma unroll
        for (int c = 0; c < 5; ++c) { const double jv = QF(rs, SMPC_REC_JDIST + p * 5 + c); rg[5 + c] += jv * nu; gd[5 + c] += jv * gam; }
      }
    }
    if (F.nn) {
      const double nu = QF(s_it, I_LAM + 21), gam = QF(s_it, I_LAM + QNR + 21);
#pragma unroll
      for (int c = 0; c < 10; ++c) { const double jv = QF(rs, SMPC_REC_JNN + c); rg[5 + c] += jv * nu; gd[5 + c] += jv * gam; }
    }
    if (k == N) {
#pragma unroll
      for (int i = 0; i < 5; ++i) { rg[i] = 0.0; gd[i] = 0.0; }
    }
    double ng = 0.0, nb = nr.nb, nd = 0.0, nm = 0.0, mu = 0.0, chk = 0.0, cnt = 0.0;
#pragma unroll
    for (int w = 0; w < PC_WARPS; ++w) {
      chk += part(w, 0);
      nm = fmax(nm, part(w, 1)); nd = fmax(nd, part(w, 2));
      ng = fmax(ng, part(w, 3)); cnt += part(w, 4);
    }
    // mu: the four partial sums in warp order, as qs_prep forms them (bit-identical results whichever form serves a problem)
    mu = ((part(0, 5) + part(1, 5)) + part(2, 5)) + part(3, 5);
#pragma unroll
    for (int i = 0; i < 15; ++i) { ng = fmax(ng, fabs(rg[i])); chk += rg[i]; if (on) QF(hc, H_GA + i) = rg[i] + gd[i]; }
    if (on) {
      double* res = q.res + qs_blk(tile, N, k, NRES, lane);
      QF(res, R_NG) = ng; QF(res, R_NB) = nb; QF(res, R_ND) = nd; QF(res, R_NM) = nm;
      QF(res, R_MU) = mu; QF(res, R_CHK) = chk; QF(res, R_CNT) = cnt;
    }
  } else {
    // ---- merge: rows of the condensed stage matrix H + reg + C' Gam C (warp 1: rows 0-8, 2: 9-11, 3: 12-14) ----
    const double hu = (k == N) ? 1.0 : QF(rs, SMPC_REC_HU) + reg;
    const double hq = QF(rs, SMPC_REC_HQ) + reg, hv = QF(rs, SMPC_REC_HV) + reg;
    // (the row loops of this phase stay unrolled: it runs after the CTA barrier, on the critical path of the work item, and rolled it loses
    // the overlap between the rows -- prep 13.4 -> 14.1 ms per cfg[1] solve, gpurun_out/r2c32)
    double Gg[12];
#pragma unroll
    for (int r = 0; r < 12; ++r) {
      const bool pres = r < 5 ? F.tau : (r < 11 ? F.dist : F.nn);
      Gg[r] = pres ? QF(s_it, I_T + 10 + r) : 0.0;
    }
    auto mrow = [&](int i) {
      double acc[15];
#pragma unroll
      for (int c = 0; c <= i; ++c) {
        double v = 0.0;
        if (c == i) v = i < 5 ? hu : ((i < 10 ? hq : hv) + QF(s_it, I_T + (i >= 5 ? i - 5 : 0)));
        if (i >= 5 && i < 10 && c >= 5) v += QF(rs, SMPC_REC_HQQ + tri(i - 5, c - 5));
        acc[c] = v;
      }
      if (F.tau) {
#pragma unroll
        for (int r = 0; r < 5; ++r) {
          const double w = Gg[r] * QF(rs, SMPC_REC_JTAU + r * 15 + i);
#pragma unroll
          for (int c = 0; c <= i; ++c) acc[c] += w * QF(rs, SMPC_REC_JTAU + r * 15 + c);
        }
      }
      if (F.dist && i >= 5 && i < 10) {
#pragma unroll
        for (int p = 0; p < 6; ++p) {
          const double w = Gg[5 + p] * QF(rs, SMPC_REC_JDIST + p * 5 + i - 5);
#pragma unroll
          for (int c = 5; c <= i; ++c) acc[c] += w * QF(rs, SMPC_REC_JDIST + p * 5 + c - 5);
        }
      }
      if (F.nn && i >= 5) {
        const double w = Gg[11] * QF(rs, SMPC_REC_JNN + i - 5);
#pragma unroll
        for (int c = 5; c <= i; ++c) acc[c] += w * QF(rs, SMPC_REC_JNN + c - 5);
      }
      if (on) {
#pragma unroll
        for (int c = 0; c <= i; ++c) QF(hc, H_M + tri(i, c)) = acc[c];
      }
    };
    if (wi == 1) {
#pragma unroll
      for (int i = 0; i < 9; ++i) mrow(i);
    } else if (wi == 2) {
#pragma unroll
      for (int i = 9; i < 12; ++i) mrow(i);
    } else {
#pragma unroll
      for (int i = 12; i < 15; ++i) mrow(i);
    }
  }
}

template <int MODE>
__global__ void __launch_bounds__(32 * SP_WARPS, QS_SP_MINB) qs_step_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int T, int kk,
                                                                                  const int* __restrict__ kk_dev) {
  if (kk_dev) kk = *kk_dev;
  const int w = blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
  if (w >= T * (q.N + 1)) return;
  qs_step(*dP, q, w / (q.N + 1), threadIdx.x & 31, w % (q.N + 1), kk, MODE);
}

// ---------------------------------------------------------------------------------------------------------------
// step, staged form: the same warp per (tile, stage) and lane per problem, and the same qs_step instruction stream per lane, with
// its operands read from a per-warp ring of SR_SLOTS chunks in shared memory instead of global memory (qp_split.cuh: QsStepGlobal,
// qs_sp).  The lowest active lane fills the ring with cp.async.bulk copies (mbarrier completion), SR_SLOTS - 1 chunks ahead of the
// arithmetic, so the loads of the next phases are in flight while a phase computes: the thread form waits for the loads of each of its
// ten phases in turn (ncu, round 2: 16 of 20 stall cycles per issue on long_scoreboard).  Slot layout = global layout, [field][lane].
// The inputs (st, st2, prod, the record, the iterate) were written by earlier kernels and nothing this kernel stores is fetched by it
// again, so no proxy fence is needed; the stores go to global memory as in the thread form.
// ---------------------------------------------------------------------------------------------------------------
constexpr int SR_SLOTS = 3;
constexpr int SR_SLOT_BYTES = qs_chunk_max_bytes();                  // 9 KB (fp64) / 7 KB (fp32 storage)
constexpr size_t SR_WARP_BYTES = ((size_t)SR_SLOTS * SR_SLOT_BYTES + 8 * SR_SLOTS + 127) / 128 * 128;   // (bulk copies: 16-byte aligned slots)
constexpr size_t SR_SMEM = SP_WARPS * SR_WARP_BYTES;
static_assert(SR_SLOT_BYTES % 128 == 0 && SR_WARP_BYTES % 128 == 0, "bulk-copy alignment");
static_assert(QS_SP_MINB * (SR_SMEM + 1024) <= 228 * 1024, "the ring keeps QS_SP_MINB CTAs per SM resident");

template <int MODE>
struct StepRing {
  unsigned char* sm;       // SR_SLOTS slots, then SR_SLOTS mbarriers
  QsBufs q;                // (kernel parameters: read from the constant bank when a copy is issued)
  size_t blk;              // tile (N + 1) + k
  const double* itp;       // iterate q.it[kk & 1]
  StageFlags F;
  unsigned mask;           // lanes that run qs_step
  int ln;
  bool lead;               // lowest lane of the mask: issues the copies
  __device__ __forceinline__ uint64_t* bar(int s) const { return reinterpret_cast<uint64_t*>(sm + (size_t)SR_SLOTS * SR_SLOT_BYTES) + s; }
  __device__ __forceinline__ const void* gsrc(const QsPiece& p) const {
    switch (p.a) {
      case QA_IT: return itp + (blk * NIT + p.f0) * TL;
      case QA_ST: return q.st + (blk * NIT + p.f0) * TL;
      case QA_ST2: return q.st2 + (blk * NS2 + p.f0) * TL;
      case QA_REC: return q.rec + (blk * REC + p.f0) * TL;
      default: return q.prod + (blk * NPROD + p.f0) * TL;
    }
  }
  __device__ __forceinline__ void issue(int c) {
    if (!lead || c >= QSC_N) return;
    const bool on = qs_chunk_on(c, F);
    const uint32_t b = smem_u32(bar(c % SR_SLOTS));
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(on ? (uint32_t)qs_chunk_bytes(MODE, c) : 0u) : "memory");
    if (!on) return;
    uint32_t dst = smem_u32(sm + (size_t)(c % SR_SLOTS) * SR_SLOT_BYTES);
#pragma unroll
    for (int i = 0; i < QSC_PIECES; ++i) {
      const QsPiece p = qs_sp(MODE, c, i);
      if (p.n == 0) continue;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(gsrc(p)),
                   "r"((uint32_t)qs_sp_bytes(p)), "r"(b) : "memory");
      dst += qs_sp_bytes(p);
    }
  }
  __device__ __forceinline__ void start() {
    if (lead) {
#pragma unroll
      for (int s = 0; s < SR_SLOTS; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar(s))));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
      for (int c = 0; c < SR_SLOTS; ++c) issue(c);
    }
    __syncwarp(mask);
  }
  __device__ __forceinline__ void acquire(int c) const {
    const uint32_t addr = smem_u32(bar(c % SR_SLOTS)), par = (uint32_t)((c / SR_SLOTS) & 1);
    uint32_t ok;
    do {
      asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(addr), "r"(par) : "memory");
    } while (!ok);
  }
  // every lane has read chunk c: its slot takes chunk c + SR_SLOTS
  __device__ __forceinline__ void release(int c) {
    __syncwarp(mask);
    issue(c + SR_SLOTS);
  }
  template <class T>
  __device__ __forceinline__ double ld(int c, int a, int f) const {
    return (double)*reinterpret_cast<const T*>(sm + (size_t)(c % SR_SLOTS) * SR_SLOT_BYTES + qs_chunk_off(MODE, c, a, f) + ln * sizeof(T));
  }
  __device__ __forceinline__ double it(int c, int f) const { return ld<double>(c, QA_IT, f); }
  __device__ __forceinline__ double st(int c, int f) const { return ld<qs_real>(c, QA_ST, f); }
  __device__ __forceinline__ double st2(int c, int f) const { return ld<qs_real>(c, QA_ST2, f); }
  __device__ __forceinline__ double prod(int c, int f) const { return ld<qs_real>(c, QA_PROD, f); }
  __device__ __forceinline__ double rec(int c, int f) const { return ld<qs_real>(c, QA_REC, f); }
};

template <int MODE>
__global__ void __launch_bounds__(32 * SP_WARPS, QS_SP_MINB) qs_step_ring_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int T, int kk,
                                                                                       const int* __restrict__ kk_dev) {
  if (kk_dev) kk = *kk_dev;
  extern __shared__ __align__(128) unsigned char sr_sm[];
  const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * SP_WARPS + wi;
  if (w >= T * (q.N + 1)) return;
  const int N = q.N, tile = w / (N + 1), k = w % (N + 1);
  const int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  const bool on = QF(pi, J_ACT) && (MODE != 2 || QF(pi, J_REDO));   // the lanes qs_step does not return from at once
  const unsigned mask = __ballot_sync(0xffffffffu, on);
  if (!on) return;
  StepRing<MODE> r;
  r.sm = sr_sm + (size_t)wi * SR_WARP_BYTES;
  r.q = q;
  r.blk = (size_t)tile * (N + 1) + k;
  r.itp = q.it[kk & 1];
  r.F = qs_flags(*dP, k);
  r.mask = mask;
  r.ln = lane;
  r.lead = lane == __ffs(mask) - 1;
  r.start();
  qs_step(*dP, q, tile, lane, k, kk, MODE, r);
}

__global__ void __launch_bounds__(32) qs_ctl_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int kk, int32_t* status, int32_t* qp_iter,
                                                     int32_t* qp_status, double* qp_res, int* counters, const int* __restrict__ kk_dev) {
  if (kk_dev) kk = *kk_dev;
  const bool on = qs_ctl<16>(*dP, q, blockIdx.x, threadIdx.x, kk, status, qp_iter, qp_status, qp_res);
  const unsigned m = __ballot_sync(0xffffffffu, on);
  if (threadIdx.x == 0 && m) atomicAdd(&counters[2 * kk], __popc(m));
}

__global__ void __launch_bounds__(32 * SP_WARPS) qs_final_kernel(QsBufs q, int T, int B, const uint8_t* __restrict__ act, int32_t* status,
                                                                 double* xt, double* ut) {
  const int w = blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
  if (w >= T * (q.N + 1)) return;
  const int tile = w / (q.N + 1), lane = threadIdx.x & 31;
  const int b = qs_final(q, tile, lane, w % (q.N + 1), act, B, status, xt, ut);
  if (b >= 0) atomicExch(&status[b], 1);
}

// ---------------------------------------------------------------------------------------------------------------
// Compaction of the slots of one tile group (qp_split.cuh: qs_compact_*).  plan: one CTA, block-wide scan over the S = 32 T
// slots -> the list of moves (active slots >= n into inactive slots < n, both in slot order: the plan of qs_compact_plan);
// move: one CTA per (move, quarter of the stages).
// ---------------------------------------------------------------------------------------------------------------
constexpr int CP_THREADS = 1024;
__global__ void __launch_bounds__(CP_THREADS) qs_compact_plan_kernel(QsBufs q, int T, int32_t* mv, int mv_half, int* n_moves) {
  __shared__ int part[CP_THREADS];
  __shared__ int s_n, s_apn;
  const int S = T * TL, tid = threadIdx.x;
  const int C = (S + CP_THREADS - 1) / CP_THREADS;
  const int s0 = tid * C, s1 = min(S, s0 + C);
  int cnt = 0;
  for (int s = s0; s < s1; ++s) {
    int32_t* pi = q.pi + qs_pb(s / TL, NPI, s % TL);
    if (QF(pi, J_ACT)) ++cnt; else QF(pi, J_FIN) = 1;          // (the results of the finished problems were written by the launch before this one)
  }
  part[tid] = cnt;
  __syncthreads();
  for (int off = 1; off < CP_THREADS; off <<= 1) {             // inclusive scan (Hillis-Steele; 1024 entries, once per compaction)
    const int v = tid >= off ? part[tid - off] : 0;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  const int before = part[tid] - cnt;                           // active slots below s0
  if (tid == CP_THREADS - 1) s_n = part[tid];
  __syncthreads();
  const int n = s_n;
  if (n >= s0 && n < s1) {                                      // the owner of slot n: actives below slot n
    int ap = before;
    for (int s = s0; s < n; ++s) ap += QF(q.pi + qs_pb(s / TL, NPI, s % TL), J_ACT) ? 1 : 0;
    s_apn = ap;
  }
  if (n >= S && tid == 0) s_apn = n;                            // every slot active: nothing moves
  __syncthreads();
  const int apn = s_apn;
  int ap = before;
  for (int s = s0; s < s1; ++s) {
    const bool a = QF(q.pi + qs_pb(s / TL, NPI, s % TL), J_ACT) != 0;
    if (a && s >= n) mv[ap - apn] = s;                          // mover number = actives in [n, s)
    if (!a && s < n) mv[mv_half + (s - ap)] = s;                // hole number = inactive slots in [0, s)
    ap += a ? 1 : 0;
  }
  if (tid == 0) *n_moves = n - apn;
}

// move: lane = move.  The plan pairs the movers (active slots beyond the boundary, in slot order) with the holes below it (in slot
// order), so 32 consecutive moves read from one or two source tiles and write into a few destination tiles: a warp instruction that
// copies one field of 32 moves touches a handful of 256-byte rows with most of their sectors in use (the first form had one thread per
// field of ONE move: every access in a row of its own, 8 useful bytes per 32-byte sector on both sides -- 1.0 -> ~0.3 ms per compaction
// of a cfg[1] solve).  CTA = four warps that take the fields of one stage of 32 moves round-robin; grid = (32-move groups, stages).
constexpr int CM_THREADS = 128;
__global__ void __launch_bounds__(CM_THREADS) qs_compact_move_kernel(QsBufs q, const int32_t* __restrict__ mv, int mv_half, const int* __restrict__ n_moves, int kk) {
  const int nm = *n_moves;
  if ((int)blockIdx.x * 32 >= nm) return;
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  if (i >= nm) return;
  const int src = mv[i], dst = mv[mv_half + i];
  const int N = q.N, k = blockIdx.y;
  const int ts = src / TL, ls = src % TL, td = dst / TL, ld = dst % TL;
  {
    const qs_real* a = q.rec + qs_blk(ts, N, k, REC, ls);
    qs_real* b = const_cast<qs_real*>(q.rec) + qs_blk(td, N, k, REC, ld);
#pragma unroll 8
    for (int f = wi; f < REC; f += CM_THREADS / 32) QF(b, f) = QF(a, f);
  }
  {
    const double* a = q.it[kk & 1] + qs_blk(ts, N, k, NIT, ls);
    double* b = q.it[kk & 1] + qs_blk(td, N, k, NIT, ld);
#pragma unroll 8
    for (int f = wi; f < NIT; f += CM_THREADS / 32) QF(b, f) = QF(a, f);
  }
  {
    const qs_real* a = q.st + qs_blk(ts, N, k, NIT, ls);
    qs_real* b = q.st + qs_blk(td, N, k, NIT, ld);
#pragma unroll 8
    for (int f = wi; f < NIT; f += CM_THREADS / 32) QF(b, f) = QF(a, f);
  }
  static_assert(CMP_FIELDS == REC + 2 * NIT, "fields of a move (qs_compact_move_field)");
  if (k == 0 && wi == 0) qs_compact_move_scalars(q, src, dst);
}


// Device warp policy of the Riccati sweeps: two staging buffers of `nfb` fields x 32 lanes in shared memory, filled by
// TMA 1-D bulk copies (cp.async.bulk global -> shared, mbarrier completion) that lane 0 issues one stage ahead.
struct TmaStage {
  qs_real* sm;
  uint64_t* bar;
  uint32_t phase[2];
  int ln, nfb;
  __device__ __forceinline__ int lane() const { return ln; }
  __device__ __forceinline__ int nbuf() const { return QS_RIC_NBUF; }
  __device__ __forceinline__ bool any(bool v) const { return __any_sync(0xffffffffu, v) != 0; }
  __device__ __forceinline__ void sync() const { __syncwarp(); }
  __device__ __forceinline__ qs_real* buf(int b) const { return sm + (size_t)b * nfb * TL + ln; }
  __device__ __forceinline__ void init() {
    phase[0] = phase[1] = 0;
    if (ln == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar + 0)));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar + 1)));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
  }
  __device__ __forceinline__ void fetch_begin(int b, int nfields) {
    if (ln == 0)
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar + b)), "r"((uint32_t)(nfields * TL * sizeof(qs_real))) : "memory");
  }
  __device__ __forceinline__ void fetch(int b, int dst_field, const qs_real* gblock, int src_field, int nfields) {
    if (ln == 0)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       smem_u32(sm + ((size_t)b * nfb + dst_field) * TL)),
                   "l"(gblock + (size_t)src_field * TL), "r"((uint32_t)(nfields * TL * sizeof(qs_real))), "r"(smem_u32(bar + b))
                   : "memory");
  }
  __device__ __forceinline__ void wait(int b) {
    const uint32_t addr = smem_u32(bar + b), par = phase[b];
    uint32_t ok;
    do {
      asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(addr), "r"(par) : "memory");
    } while (!ok);
    phase[b] = par ^ 1u;
  }
  // hint: start moving a field range of a stage block towards L2
  __device__ __forceinline__ void prefetch(const qs_real* gblock, int src_field, int nfields) const {
    if (ln == 0)
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gblock + (size_t)src_field * TL), "r"((uint32_t)(nfields * TL * sizeof(qs_real))) : "memory");
  }
  // this lane's global stores become visible to bulk copies issued after the next warp barrier
  __device__ __forceinline__ void publish() const { asm volatile("fence.proxy.async;" ::: "memory"); }
};

constexpr size_t RIC1_SMEM = sizeof(double) * 65 * TL + sizeof(qs_real) * (QS_RIC_NBUF * RIC1_STAGE_FIELDS) * TL + 16;   // P scratch (fp64) + staging
constexpr size_t RIC2_SMEM = sizeof(qs_real) * (QS_RIC_NBUF * RIC2_STAGE_FIELDS) * TL + 16;

__global__ void __launch_bounds__(32) qs_ric1_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q) {
  extern __shared__ __align__(128) double smem[];
  TmaStage w;
  double* psm = smem;                                        // P_{k+1}, p_{k+1}: on-chip only, fp64 in both flavours
  w.sm = reinterpret_cast<qs_real*>(psm + 65 * TL); w.nfb = RIC1_STAGE_FIELDS; w.ln = threadIdx.x;
  w.bar = reinterpret_cast<uint64_t*>(w.sm + (size_t)QS_RIC_NBUF * RIC1_STAGE_FIELDS * TL);
  w.init();
  qs_ric1(*dP, q, blockIdx.x, w, psm + threadIdx.x);
}

// ---------------------------------------------------------------------------------------------------------------
// ric1, two warps per tile (lane = problem in both).  The sweep is a dependent instruction stream of ~2 000 instructions per
// stage that a single warp issues at the latency of its FP64 chains (profiles/r01_qp_v7.md), so its duration -- the same for 1 or
// 10 000 active problems -- is cut by splitting the stream, not by adding tiles:
//   warp A (control columns):  y = P_{k+1} rb + p_{k+1}, gradient, the 15 x 5 panel, its LDL' elimination -> T, l~, p_k
//   warp B (state block):      trailing base  M_xx + [A]' P_{k+1} [A]  for the 55 entries of the state block while A eliminates,
//                              then  P_k = base - T_x D T_x'  once A has published T_x and D through shared memory
// Two named barriers per stage (T published / P_k complete).  The staging buffer is released at the first barrier, so the TMA
// fetch of the next stage runs under B's second half and A's stores.  Stage 0: B factorises P_0, solves for dx_0 and runs the
// forward substitution with two staging buffers (the P scratch is free by then); A has exited.
// Per-entry arithmetic and summation order are those of qs_ric1 (qp_split.cuh): results are bit-identical.
// ---------------------------------------------------------------------------------------------------------------
constexpr int R1X_XF = 55;                                                     // exchange: T rows 5-14 (50) + D (5)
constexpr int R1X_FIELDS = RIC1_STAGE_FIELDS + 65 + R1X_XF;                    // 265
constexpr int R1X_FWD = B_WV - B_RB;                                           // forward stage fetch: RB LP T (100 fields)
constexpr int R1X_FWD1 = 136;                                                  // field offset of the second forward buffer
static_assert(R1X_FWD1 >= R1X_FWD && R1X_FWD1 + R1X_FWD <= R1X_FIELDS, "forward buffers");
// bytes: backward staging [B_M, B_LP) in the storage type, then P / p scratch and the exchange block in fp64; the two forward buffers
// overlay the front of it (the scratch is free by then)
constexpr size_t R1X_STG_BYTES = sizeof(qs_real) * RIC1_STAGE_FIELDS * TL;
constexpr size_t R1X_BYTES = R1X_STG_BYTES + sizeof(double) * (65 + R1X_XF) * TL;
static_assert(sizeof(qs_real) * (R1X_FWD1 + R1X_FWD) * TL <= R1X_BYTES, "forward buffers");
constexpr size_t RIC1X_SMEM = R1X_BYTES + 32;

// named barrier of the two warps of a tile.  The warps reach it from different code paths and, inside a warp, lanes may arrive from a
// data-dependent branch (a non-positive pivot, an inactive lane): the warp reconverges first and the barrier is the non-aligned form
// (bar.sync = barrier.sync.aligned is undefined for a diverged warp; compute-sanitizer synccheck flagged it, gpurun_out/r2c17)
__device__ __forceinline__ void r1x_bar() {
  __syncwarp();
  asm volatile("barrier.sync 1, 64;" ::: "memory");
}
__device__ __forceinline__ void r1x_fetch(qs_real* dst, const qs_real* src, int nfields, uint64_t* bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"((uint32_t)(nfields * TL * sizeof(qs_real))) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"((uint32_t)(nfields * TL * sizeof(qs_real))), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void r1x_wait(uint64_t* bar, uint32_t& phase) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(addr), "r"(phase) : "memory");
  } while (!ok);
  phase ^= 1u;
}

__global__ void __launch_bounds__(64) qs_ric1x_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q) {
  extern __shared__ __align__(128) double smem[];
  const smpc_problem_t& P = *dP;
  const int N = q.N, tile = blockIdx.x, lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  const bool on = QF(pi, J_ACT) != 0;
  if (!__any_sync(0xffffffffu, on)) return;                 // (both warps: same tile, same answer)
  qs_real* stg_all = reinterpret_cast<qs_real*>(smem);       // backward staging: fields [B_M, B_LP) at their own offsets
  double* psm_all = reinterpret_cast<double*>(reinterpret_cast<char*>(smem) + R1X_STG_BYTES);   // P_{k+1} (55) and p_{k+1} (10), fp64
  double* xch_all = psm_all + (size_t)65 * TL;               // T rows 5-14 and D of the running stage, fp64
  uint64_t* bar = reinterpret_cast<uint64_t*>(reinterpret_cast<char*>(smem) + R1X_BYTES);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar + 0)));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar + 1)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  double* pd = q.pd + qs_pb(tile, NPD, lane);
  const double dt = P.dt, a2 = 0.5 * P.dt * P.dt;
  const qs_real* gsb = q.sb + qs_blk(tile, N, 0, NSB, 0);
  const size_t sstride = (size_t)NSB * TL;
  const qs_real* hc = stg_all + lane;
  double* psm = psm_all + lane;
  double* xch = xch_all + lane;
  auto Pn = [&](int idx) { return QF(psm, idx); };
  uint32_t ph0 = 0;
  if (threadIdx.x == 0) r1x_fetch(stg_all, gsb + (size_t)N * sstride + (size_t)B_M * TL, B_LP - B_M, bar);
  double dx[10];
#pragma unroll
  for (int i = 0; i < 10; ++i) dx[i] = 0.0;

  for (int k = N; k >= 0; --k) {
    r1x_wait(bar, ph0);
    qs_real* fac = q.sb + qs_blk(tile, N, k, NSB, lane);
    if (wi == 0) {
      // ---------------- warp A: gradient, panel, elimination ----------------
      double g[15];
#pragma unroll
      for (int i = 0; i < 15; ++i) g[i] = QF(hc, H_GA + i);
      if (k < N) {
        double rb[10], y[10];
#pragma unroll
        for (int j = 0; j < 10; ++j) rb[j] = QF(hc, H_RB + j);
#pragma unroll
        for (int i = 0; i < 10; ++i) {
          double s = 0.0;
#pragma unroll
          for (int j = 0; j < 10; ++j) s += Pn(trs(i, j)) * rb[j];
          if (on) QF(fac, F_WV + i) = s;
          y[i] = s + QF(psm, 55 + i);
        }
#pragma unroll
        for (int j = 0; j < 5; ++j) {
          g[j] += a2 * y[j] + dt * y[5 + j];
          g[5 + j] += y[j];
          g[10 + j] += dt * y[j] + y[5 + j];
        }
      } else {
#pragma unroll
        for (int i = 0; i < 5; ++i) g[i] = 0.0;
      }
      double pan[15][5];
#pragma unroll
      for (int i = 0; i < 15; ++i)
#pragma unroll
        for (int j = 0; j < 5; ++j)
          if (j <= i) pan[i][j] = QF(hc, H_M + tri(i, j)) + (k < N ? qs_y(i, j, dt, a2, Pn) : 0.0);
      double dd[5];
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const double d = pan[j][j];
        const double invd = d > 0.0 ? qs_rcp(d) : 0.0;
        dd[j] = d > 0.0 ? d : 0.0;
#pragma unroll
        for (int i = 14; i > j; --i) {
          const double t = pan[i][j] * invd;
          g[i] -= t * g[j];
#pragma unroll
          for (int c = j + 1; c < 5; ++c)
            if (c <= i) pan[i][c] -= t * pan[c][j];
          pan[i][j] = t;
        }
        pan[j][j] = invd;
      }
#pragma unroll
      for (int i = 5; i < 15; ++i)
#pragma unroll
        for (int j = 0; j < 5; ++j) QF(xch, (i - 5) * 5 + j) = pan[i][j];
#pragma unroll
      for (int j = 0; j < 5; ++j) QF(xch, 50 + j) = dd[j];
#pragma unroll
      for (int i = 0; i < 10; ++i) QF(psm, 55 + i) = g[5 + i];           // p_k (read by A at the next stage, by B at stage 0)
      r1x_bar();                                                          // (1) T_x, D published; staging buffer free
      if (lane == 0 && k > 0) r1x_fetch(stg_all, gsb + (size_t)(k - 1) * sstride + (size_t)B_M * TL, B_LP - B_M, bar);
      if (on) {
#pragma unroll
        for (int i = 0; i < 15; ++i)
#pragma unroll
          for (int j = 0; j < 5; ++j)
            if (j <= i) QF(fac, F_T + i * 5 + j) = pan[i][j];
#pragma unroll
        for (int i = 0; i < 15; ++i) QF(fac, F_LP + i) = g[i];
      }
      if (k == 0) asm volatile("fence.proxy.async;" ::: "memory");       // T, l~ of every stage visible to the bulk copies of the forward sweep
      r1x_bar();                                                          // (2) P_k complete
    } else {
      // ---------------- warp B: state block ----------------
      double tb[10][10];
#pragma unroll
      for (int i = 5; i < 15; ++i)
#pragma unroll
        for (int c = 5; c <= i; ++c) tb[i - 5][c - 5] = QF(hc, H_M + tri(i, c)) + (k < N ? qs_y(i, c, dt, a2, Pn) : 0.0);
      r1x_bar();                                                          // (1)
#pragma unroll
      for (int i = 5; i < 15; ++i) {
        double sdx[5];
#pragma unroll
        for (int j = 0; j < 5; ++j) sdx[j] = QF(xch, (i - 5) * 5 + j) * QF(xch, 50 + j);
#pragma unroll
        for (int c = 5; c <= i; ++c) {
          double v = tb[i - 5][c - 5];
#pragma unroll
          for (int j = 0; j < 5; ++j) v -= sdx[j] * QF(xch, (c - 5) * 5 + j);
          tb[i - 5][c - 5] = v;
        }
      }
#pragma unroll
      for (int i = 0; i < 10; ++i)
#pragma unroll
        for (int c = 0; c <= i; ++c) { QF(psm, tri(i, c)) = tb[i][c]; if (on) QF(fac, F_P + tri(i, c)) = tb[i][c]; }
      if (k == 0) {
        // factorise P_0 (kept per problem for the re-solves of ric2) and solve P_0 dx_0 = -p_0
        double gg[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) gg[i] = QF(psm, 55 + i);
#pragma unroll
        for (int j = 0; j < 10; ++j) {
          const double d = tb[j][j];
          const double invd = d > 0.0 ? qs_rcp(d) : 0.0;
          tb[j][j] = invd;
#pragma unroll
          for (int i = 9; i > j; --i) {
            const double t = tb[i][j] * invd;
            gg[i] -= t * gg[j];
#pragma unroll
            for (int c = j + 1; c <= i; ++c) tb[i][c] -= t * tb[c][j];
            tb[i][j] = t;
          }
        }
        if (on) {
#pragma unroll
          for (int i = 0; i < 10; ++i)
#pragma unroll
            for (int c = 0; c <= i; ++c) QF(pd, D_T0 + tri(i, c)) = tb[i][c];
        }
#pragma unroll
        for (int i = 9; i >= 0; --i) {
          double acc = tb[i][i] * gg[i];
#pragma unroll
          for (int c = i + 1; c < 10; ++c) acc += tb[c][i] * dx[c];
          dx[i] = tb[i][i] > 0.0 ? -acc : 0.0;
        }
      }
      r1x_bar();                                                          // (2)
    }
  }
  if (wi == 0) return;

  // ---------------- warp B: forward substitution (affine direction), two staging buffers ----------------
  uint32_t ph[2] = {ph0, 0};
  qs_real* fb[2] = {stg_all, stg_all + (size_t)R1X_FWD1 * TL};
  if (lane == 0) r1x_fetch(fb[0], gsb + (size_t)B_RB * TL, R1X_FWD, bar + 0);
  for (int k = 0; k <= N; ++k) {
    __syncwarp();                                                          // every lane is done with the buffer of stage k - 1
    if (lane == 0 && k < N) r1x_fetch(fb[(k + 1) & 1], gsb + (size_t)(k + 1) * sstride + (size_t)B_RB * TL, R1X_FWD, bar + ((k + 1) & 1));
    r1x_wait(bar + (k & 1), ph[k & 1]);
    const qs_real* sb = fb[k & 1] + lane - (size_t)B_RB * TL;              // sb[f] valid for B_RB <= f < B_WV
    qs_real* st = q.st + qs_blk(tile, N, k, NIT, lane);
    double du[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) du[i] = 0.0;
    if (k < N) {
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        double ws = (double)QF(sb, F_T + i * 5 + i) * (double)QF(sb, F_LP + i);   // (operands widened first: fp32-storage flavour)
#pragma unroll
        for (int r = 0; r < 10; ++r) ws += QF(sb, F_T + (5 + r) * 5 + i) * dx[r];
        du[i] = -ws;
      }
#pragma unroll
      for (int c = 4; c >= 1; --c)
#pragma unroll
        for (int i = 0; i < c; ++i) du[i] -= QF(sb, F_T + c * 5 + i) * du[c];
    }
    if (on) {
#pragma unroll
      for (int i = 0; i < 5; ++i) QF(st, I_Z + i) = du[i];
#pragma unroll
      for (int i = 0; i < 10; ++i) QF(st, I_Z + 5 + i) = dx[i];
    }
    if (k < N) {
      double nx[10];
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        nx[j] = dx[j] + dt * dx[5 + j] + a2 * du[j] + QF(sb, H_RB + j);
        nx[5 + j] = dx[5 + j] + dt * du[j] + QF(sb, H_RB + 5 + j);
      }
#pragma unroll
      for (int j = 0; j < 10; ++j) dx[j] = nx[j];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Tail kernels: one WARP per problem (the sweeps themselves: qp_tail.cuh).  One CTA serves RT_WARPS problems of a tile; warps of
// finished problems exit at once.
// ---------------------------------------------------------------------------------------------------------------
#include "qp_tail.cuh"

__global__ void __launch_bounds__(32 * RT_WARPS) qs_ric1t_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q) {
  extern __shared__ __align__(16) unsigned char rt_sm[];
  const int tile = blockIdx.x / (32 / RT_WARPS), wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pl = (blockIdx.x % (32 / RT_WARPS)) * RT_WARPS + wi;          // problem (lane of the tile) this warp serves
  if (!QF(q.pi + qs_pb(tile, NPI, pl), J_ACT)) return;
  double* W = reinterpret_cast<double*>(rt_sm + (size_t)wi * RT_WARP_BYTES);
  rt_ric1(*dP, q, tile, pl, lane, W, reinterpret_cast<qs_real*>(W + RT_WORK));
}

__global__ void __launch_bounds__(32 * RT_WARPS) qs_ric2t_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q) {
  extern __shared__ __align__(16) unsigned char rt_sm[];
  const int tile = blockIdx.x / (32 / RT_WARPS), wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pl = (blockIdx.x % (32 / RT_WARPS)) * RT_WARPS + wi;
  if (!QF(q.pi + qs_pb(tile, NPI, pl), J_ACT)) return;
  double* W = reinterpret_cast<double*>(rt_sm + (size_t)wi * RT_WARP_BYTES);
  rt_ric2(*dP, q, tile, pl, lane, W, reinterpret_cast<qs_real*>(W + RT_WORK));
}

// ---------------------------------------------------------------------------------------------------------------
// Solo kernel: one CTA per problem runs WHOLE interior-point iterations on the device until its problem has finished -- no
// launch per phase, no counter read-back, nobody waits for anybody else.  Used (a) for the tail of a solve, once at most
// `solo_max` problems of a tile group still iterate (a problem that runs into qp_max_iter used to hold the batch for ~190
// iterations of ~9 launches each), and (b) from the first iteration on for small batches (configs[0]: 100 problems, less than one
// problem per SM), where a solve is nothing but latency.  The phases are the functions of qp_split.cuh and the warp-per-problem
// sweeps above, on the same arrays (a problem's working set, ~340 KB, lives in L2), separated by CTA barriers: thread k serves
// stage k in the stage-parallel phases, warp 0 runs the sweeps, thread 0 the per-problem control logic.  Same functions, same
// operands: results are bit-identical to the multi-kernel path, so a problem's result does not depend on who served it.
// ---------------------------------------------------------------------------------------------------------------
constexpr int SOLO_THREADS = 64;
constexpr size_t SOLO_SMEM = sizeof(double) * (SOLO_THREADS / 32) * PREP_SCRATCH * TL + RT_WARP_BYTES + 16;

__global__ void __launch_bounds__(SOLO_THREADS) qs_solo_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int kk0, int32_t* status, int32_t* qp_iter,
                                                               int32_t* qp_status, double* qp_res) {
  extern __shared__ __align__(16) double so_sm[];
  __shared__ int s_on, s_redo;
  const smpc_problem_t& P = *dP;
  const int N = q.N, tile = blockIdx.x / TL, pl = blockIdx.x % TL, tid = threadIdx.x, lane = tid & 31, wi = tid >> 5;
  int32_t* pi = q.pi + qs_pb(tile, NPI, pl);
  if (!QF(pi, J_ACT)) return;                                // (the whole CTA: same slot)
  double* jsm = so_sm + (size_t)wi * PREP_SCRATCH * TL + lane;
  double* W = so_sm + (size_t)(SOLO_THREADS / 32) * PREP_SCRATCH * TL;
  qs_real* ring = reinterpret_cast<qs_real*>(W + RT_WORK);
#ifdef QS_SOLO_TIMING
  long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t0 = clock64(), t1;
  int nit = 0;
#define SOLO_T(i) { t1 = clock64(); tph[i] += t1 - t0; t0 = t1; }
#else
#define SOLO_T(i)
#endif
  for (int kk = kk0;; ++kk) {
    if (tid == 0) s_on = qs_ctl(P, q, tile, pl, kk, status, qp_iter, qp_status, qp_res) ? 1 : 0;
    __syncthreads();
    SOLO_T(0)
    if (!s_on) break;
    if (wi == 0) rt_ric1(P, q, tile, pl, lane, W, ring);
    __syncthreads();
    SOLO_T(1)
    for (int k = tid; k <= N; k += SOLO_THREADS) qs_step(P, q, tile, pl, k, kk, 0);
    __syncthreads();
    SOLO_T(2)
    if (wi == 0) rt_ric2(P, q, tile, pl, lane, W, ring);
    __syncthreads();
    SOLO_T(3)
    for (int k = tid; k <= N; k += SOLO_THREADS) qs_step(P, q, tile, pl, k, kk, 1);
    __syncthreads();
    SOLO_T(4)
    if (tid == 0) { qs_red(P, q, tile, pl, false); s_redo = QF(pi, J_REDO); }
    __syncthreads();
    SOLO_T(5)
    if (s_redo) {
      for (int k = tid; k <= N; k += SOLO_THREADS) qs_step(P, q, tile, pl, k, kk, 2);
      __syncthreads();
      if (tid == 0) qs_red(P, q, tile, pl, true);
      __syncthreads();
    }
    SOLO_T(6)
    for (int k = tid; k <= N; k += SOLO_THREADS) qs_prep<false>(P, q, tile, pl, k, kk + 1, jsm);
    __syncthreads();
    SOLO_T(7)
#ifdef QS_SOLO_TIMING
    ++nit;
#endif
  }
#ifdef QS_SOLO_TIMING
  if (tid == 0 && blockIdx.x < 2 && nit > 0)
    printf("SOLO slot %d its %d cycles/it: ctl %lld ric1 %lld step0 %lld ric2 %lld step1 %lld red %lld redo %lld prep %lld\n", blockIdx.x, nit, tph[0] / nit,
           tph[1] / nit, tph[2] / nit, tph[3] / nit, tph[4] / nit, tph[5] / nit, tph[6] / nit, tph[7] / nit);
#endif
}

__global__ void __launch_bounds__(32) qs_ric2_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q) {
  extern __shared__ __align__(128) double smem[];
  TmaStage w;
  w.sm = reinterpret_cast<qs_real*>(smem); w.nfb = RIC2_STAGE_FIELDS; w.ln = threadIdx.x;
  w.bar = reinterpret_cast<uint64_t*>(w.sm + (size_t)QS_RIC_NBUF * RIC2_STAGE_FIELDS * TL);
  w.init();
  qs_ric2(*dP, q, blockIdx.x, w);
}

// redo_list: the slots (of this group) whose problem fell back to the centering direction, tile by tile in arrival order of the tiles
__global__ void __launch_bounds__(32) qs_red_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int kk, int after_redo, int* counters, int32_t* redo_list,
                                                    const int* __restrict__ kk_dev) {
  if (kk_dev) kk = *kk_dev;
  qs_red(*dP, q, blockIdx.x, threadIdx.x, after_redo != 0);
  if (!after_redo) {
    const int32_t* pi = q.pi + qs_pb(blockIdx.x, NPI, threadIdx.x);
    const bool redo = QF(pi, J_ACT) && QF(pi, J_REDO);
    const unsigned m = __ballot_sync(0xffffffffu, redo);
    int base = 0;
    if (threadIdx.x == 0 && m) base = atomicAdd(&counters[2 * kk + 1], __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (redo) redo_list[base + __popc(m & ((1u << threadIdx.x) - 1u))] = blockIdx.x * TL + threadIdx.x;
  }
}

// Device-side loop of a solve captured into a CUDA graph (qp_split.cuh: qs_graph_drive), one thread each.  reset: every launch of the
// graph starts a fresh solve at iteration 0 and enters the loop body;  loop: the loop step of qs_loop_step sets the condition of the
// WHILE node that repeats the body.
__global__ void __launch_bounds__(1) qs_loop_reset_kernel(int* kk_dev, cudaGraphConditionalHandle cond) {
  *kk_dev = 0;
  cudaGraphSetConditional(cond, 1);
}
__global__ void __launch_bounds__(1) qs_loop_kernel(const int* __restrict__ counters, int* kk_dev, int iter_max, cudaGraphConditionalHandle cond) {
  cudaGraphSetConditional(cond, qs_loop_step(counters, kk_dev, iter_max) ? 1u : 0u);
}

// The switch to the centering direction for FEW flagged problems: one CTA per list entry, thread = stage (qs_step mode 2), then thread 0
// takes the step length of the new direction (qs_red, second call) -- the same two functions as the launches qs_step_kernel<2> + qs_red_kernel
// they replace, on the same operands (bit-identical), but the work is proportional to the number of flagged PROBLEMS: the tile form runs a
// whole warp for every (tile, stage) that holds at least one flagged lane, i.e. nearly all of them once 5 % of the problems are flagged.
constexpr int RL_THREADS = 64;
__global__ void __launch_bounds__(RL_THREADS) qs_redo_list_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int kk, const int32_t* __restrict__ redo_list,
                                                                  const int* __restrict__ n_list) {
  if ((int)blockIdx.x >= *n_list) return;
  const int slot = redo_list[blockIdx.x], tile = slot / TL, pl = slot % TL;
  for (int k = threadIdx.x; k <= q.N; k += RL_THREADS) qs_step(*dP, q, tile, pl, k, kk, 2);
  __syncthreads();
  if (threadIdx.x == 0) qs_red(*dP, q, tile, pl, true);
}

// stage records, tile-interleaved -> caller layout [B][N+1][REC] (smpc_get_lin)
__global__ void rec_untile_kernel(int B, int N, const qs_real* __restrict__ rec, double* out) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * (N + 1) * REC) return;
  const int f = idx % REC;
  const size_t bk = idx / REC;
  const int k = bk % (N + 1), b = bk / (N + 1);
  out[idx] = QF(rec + qs_blk(b / TL, N, k, REC, b % TL), f);
}

// canonical dump of the QP solution for parity tests (layout of smpc_get_qp)
__global__ void dump_qp_kernel(const smpc_problem_t* __restrict__ dP, QsBufs q, int B, double* dz, double* pi, double* lam, double* t) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int N = q.N;
  if (idx >= B * (N + 1)) return;
  const int b = idx / (N + 1), k = idx % (N + 1);
  const int tile = b / TL, lane = b % TL;
  const int buf = QF(q.pi + qs_pb(tile, NPI, lane), J_ITBUF);
  const double* it = q.it[buf] + qs_blk(tile, N, k, NIT, lane);
  const StageFlags F = qs_flags(*dP, k);
  if (dz) {
    double* o = dz + (size_t)idx * 15;
    if (k < N) for (int i = 0; i < 15; ++i) o[i] = QF(it, I_Z + i);
    else { for (int i = 0; i < 10; ++i) o[i] = QF(it, I_Z + 5 + i); for (int i = 10; i < 15; ++i) o[i] = 0.0; }
  }
  if (pi && k > 0) for (int i = 0; i < 10; ++i) pi[((size_t)b * N + k - 1) * 10 + i] = QF(it, I_PIM + i);
  if (lam && t) {
    double* ol = lam + (size_t)idx * SMPC_QP_NC;
    double* ot = t + (size_t)idx * SMPC_QP_NC;
    for (int j = 0; j < QNR; ++j) {
      const bool p = j < 10 ? true : (j < 15 ? F.tau : (j < 21 ? F.dist : F.nn));
      for (int s = 0; s < 2; ++s) { ol[s * QNR + j] = p ? QF(it, I_LAM + s * QNR + j) : 0.0; ot[s * QNR + j] = p ? QF(it, I_T + s * QNR + j) : 0.0; }
    }
    ol[2 * QNR] = F.soft ? QF(it, I_SLK + 2) : 0.0; ol[2 * QNR + 1] = F.soft ? QF(it, I_SLK + 3) : 0.0;
    ot[2 * QNR] = F.soft ? QF(it, I_SLK + 4) : 0.0; ot[2 * QNR + 1] = F.soft ? QF(it, I_SLK + 5) : 0.0;
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------ solver object
#ifndef QS_GROUPS
#define QS_GROUPS 1              // tile groups solved concurrently on their own streams (see QsLoop).  Round 1 ran three (the latency-bound sweeps of one
                                 // group under the streaming kernels of the others: +3 %); since the slots are compacted between iterations and every
                                 // kernel runs at 0.6-0.95 of the HBM peak on the full batch, one group is faster: cfg[1] 60.25 -> 59.38 ms per step, cfg[2]
                                 // HTWA 33.45 -> 32.29 ms (three runs each, gpurun_out/r2tune, r2tune2); SMPC_QP_GROUPS=n brings the groups back
#endif
constexpr int MAX_GROUPS = 8;
constexpr int RING = 8;          // counter read-backs in flight per group (run-ahead depth + 2 at most)

// optional timeline (profiling / SMPC_QP_TRACE=1): one event pair per kernel
struct TraceRec { int g; const char* name; int kk; cudaEvent_t a, b; };

struct QpGroup {
  QsBufs q{};
  int T = 0;                    // tiles of this group
  cudaStream_t stream = nullptr;   // stage-parallel kernels (bandwidth-bound)
  cudaStream_t hi = nullptr;       // Riccati sweeps (latency-bound, few warps): higher priority, so that their CTAs take the
                                   // slots that retiring stage-parallel CTAs of the other groups free
  cudaEvent_t ev[RING] = {nullptr};   // ev[kk % RING]: the counters of iteration kk have landed in h_counters[2 (kk % RING)]
  cudaEvent_t ev_done = nullptr;      // last kernel of the solve
  cudaEvent_t evx = nullptr;    // hand-over between the two streams
  int* counters = nullptr;      // [2 (iter_max + 2)]: active / redo per IPM iteration
  int* h_counters = nullptr;    // pinned, 2 RING ints
  int32_t* mv = nullptr;        // compaction: [2][mv_half] source / destination slots
  int mv_half = 0;
  int* n_moves = nullptr;       // device
  int32_t* redo_list = nullptr; // [32 T] slots flagged for the centering direction in the current iteration (qs_red_kernel)
  int in_use = 0;               // slots that may still hold an iterating problem (32 T at the start of a solve, less after a compaction)
  int* kk_dev = nullptr;        // IPM iteration of a solve captured into a graph (device)
  cudaStream_t body = nullptr;  // captures the loop body of such a solve
  int tiles() const { return (in_use + TL - 1) / TL; }
};

struct QpSolver {
  int B = 0, N = 0, T = 0, iter_max = 0, G = 1;
  QsBufs q{};                   // whole batch (group 0 .. G-1 are sub-ranges of its tiles)
  QpGroup grp[MAX_GROUPS];
  double* block = nullptr;      // one allocation for all arrays: the fp64 ones first, then the ones of the storage type
  int32_t* pi = nullptr;
  int* counters = nullptr;
  int* h_counters = nullptr;
  int* kk_dev = nullptr;        // [G]
  int32_t* mv = nullptr;        // compaction plans of the groups
  int* n_moves = nullptr;
  int32_t* redo_list = nullptr;
  int redo_list_max = -1;       // the centering switch runs one CTA per flagged problem when at most this many are flagged (-1: an eighth of the slots in
                                // use; 0: never; SMPC_QP_REDO_LIST).  Measured on cfg[1] (gpurun_out/r2c25, 3 runs each): never 57.8 ms per step, 1/8 57.5,
                                // 1/4 57.9, 1/2 58.8 -- the list kernel (254 registers, lane-strided accesses) only pays for a few hundred problems
  cudaEvent_t ev_in = nullptr;  // inputs (records, x0) are ready on the caller's stream
  int last_iters = 0;
  int solo_max = 384;           // a solve of at most this many problems per tile group is run by the solo kernel (one CTA per problem, whole iterations on
                                // the device, one launch per solve; SMPC_QP_SOLO; 0: never)
  bool solo_tail = false;       // ... and so is the tail of a larger solve once that few problems are left (SMPC_QP_SOLO_TAIL=1).  Off: measured on B200
                                // (profiles/r02_solo.md) a solo iteration takes 0.42 ms against 0.23 ms for a tail iteration of the multi-kernel path
  int tail_max = 384;           // a tile group with at most this many problems still iterating is served by the warp-per-problem sweeps (0: never)
  int tail_which = 3;           // development: bit 0 / 1 = the factorising / the vector sweep may use the warp-per-problem form (SMPC_QP_TAIL_WHICH)
  bool split_ric1 = true;       // two warps per tile in the factorising Riccati sweep (SMPC_QP_RIC1=single selects the one-warp form)
  bool coop_prep = true;        // kk >= 1: four-warp cooperative prep with TMA-staged inputs (SMPC_QP_PREP=thread selects the thread-per-stage form)
  bool ring_step = true;        // step kernels read their operands from a per-warp ring of bulk copies (SMPC_QP_STEP=thread: straight from global memory)
  bool profile = false;         // record one event pair per kernel of the next solves (smpc_set_profiling)
  double prof_ms[SMPC_PROF_N] = {0};
  int32_t prof_n[SMPC_PROF_N] = {0};
  double prof_span_ms = 0.0;
  int depth = 0;                // IPM iterations the host queues ahead of the counters it has seen (SMPC_QP_DEPTH).  Default 0 = one round trip per
                                // iteration: measured on B200 (profiles/r02_qp_loop.md) running ahead costs two unconditional launches per iteration
                                // (step<2>, red) and gains nothing while three tile groups already cover the round trip
  bool compact = true;          // pack the problems still iterating into the leading slots between iterations (SMPC_QP_COMPACT=0: never)
  int compact_min_tiles = 32;   // ... for groups of at least this many tiles
  double compact_at = 0.85;     // ... once the active count has fallen to this fraction of the slots in use (SMPC_QP_COMPACT_AT)
  bool compacted = false;       // the last solve reused slots: per-slot dumps (smpc_get_lin / smpc_get_qp) are not available for it
  int n_compactions = 0;        // of the last solve
  bool trace_print = false;     // SMPC_QP_TRACE=1
  std::vector<struct TraceRec> trace;   // optional timeline: one event pair per kernel (profiling / SMPC_QP_TRACE)
};

size_t qp_bytes(int B, int N) {
  const size_t T = (B + TL - 1) / TL, S = T * (N + 1) * TL;
  return sizeof(double) * (S * (2 * NIT + NRES + NSTP) + T * NPD * TL) + sizeof(qs_real) * S * (REC + NIT + NS2 + NSB + NPROD);
}

QpSolver* qp_create(int B, int N, int iter_max, bool keep_slots, cudaStream_t stream, cudaError_t* err) {
  QpSolver* s = new QpSolver;
  s->B = B; s->N = N; s->T = (B + TL - 1) / TL; s->iter_max = iter_max;
  const size_t T = s->T, S = T * (N + 1) * TL;
  // groups: at least ~64 tiles each so that the stage-parallel kernels of one group still fill the GPU
  int G = QS_GROUPS;
  if (const char* e = getenv("SMPC_QP_GROUPS")) G = atoi(e);
  while (G > 1 && s->T / G < 64) --G;
  if (G < 1) G = 1;
  if (G > MAX_GROUPS) G = MAX_GROUPS;
  s->G = G;
  const size_t ncnt = (size_t)2 * (iter_max + 2);
  cudaError_t e = cudaMalloc((void**)&s->block, qp_bytes(B, N));
  if (e == cudaSuccess) e = cudaMemsetAsync(s->block, 0, qp_bytes(B, N), stream);
  if (e == cudaSuccess) e = cudaMalloc((void**)&s->pi, sizeof(int32_t) * T * NPI * TL);
  if (e == cudaSuccess) e = cudaMemsetAsync(s->pi, 0, sizeof(int32_t) * T * NPI * TL, stream);
  if (e == cudaSuccess) e = cudaMalloc((void**)&s->counters, sizeof(int) * ncnt * G);
  if (e == cudaSuccess) e = cudaMallocHost((void**)&s->h_counters, sizeof(int) * 2 * RING * G);
  if (e == cudaSuccess) e = cudaMalloc((void**)&s->kk_dev, sizeof(int) * G);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_in, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaMalloc((void**)&s->mv, sizeof(int32_t) * ((size_t)s->T * TL + 2 * MAX_GROUPS));
  if (e == cudaSuccess) e = cudaMalloc((void**)&s->n_moves, sizeof(int) * MAX_GROUPS);
  if (e == cudaSuccess) e = cudaMalloc((void**)&s->redo_list, sizeof(int32_t) * (size_t)s->T * TL);
  if (const char* pe = getenv("SMPC_QP_REDO_LIST")) s->redo_list_max = atoi(pe);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_prep_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PREP_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_prep_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PREP_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_prep_coop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PC_SMEM);
  if (const char* pe = getenv("SMPC_QP_PREP")) s->coop_prep = strcmp(pe, "thread") != 0;
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_step_ring_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SR_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_step_ring_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SR_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_step_ring_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SR_SMEM);
  if (const char* se = getenv("SMPC_QP_STEP")) s->ring_step = strcmp(se, "thread") != 0;
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_ric1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RIC1_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_ric1x_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RIC1X_SMEM);
  if (const char* re = getenv("SMPC_QP_RIC1")) s->split_ric1 = strcmp(re, "single") != 0;
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_ric1t_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_ric2t_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_SMEM);
  if (const char* te = getenv("SMPC_QP_TAIL")) s->tail_max = atoi(te);
  if (const char* te = getenv("SMPC_QP_TAIL_WHICH")) s->tail_which = atoi(te);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_solo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SOLO_SMEM);
  if (const char* se = getenv("SMPC_QP_SOLO")) s->solo_max = atoi(se);
  if (const char* se = getenv("SMPC_QP_SOLO_TAIL")) s->solo_tail = atoi(se) != 0;
  if (const char* de = getenv("SMPC_QP_DEPTH")) s->depth = atoi(de);
  if (s->depth < 0) s->depth = 0;
  if (s->depth > RING - 2) s->depth = RING - 2;
  if (const char* ce = getenv("SMPC_QP_COMPACT")) s->compact = atoi(ce) != 0;
  if (const char* ce = getenv("SMPC_QP_COMPACT_AT")) { const double v = atof(ce); if (v > 0.1 && v < 1.0) s->compact_at = v; }
  if (keep_slots) s->compact = false;
  s->trace_print = getenv("SMPC_QP_TRACE") != nullptr;
  if (e == cudaSuccess) e = cudaFuncSetAttribute(qs_ric2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RIC2_SMEM);
  for (int g = 0; g < G && e == cudaSuccess; ++g) {
    int plo = 0, phi = 0;
    cudaDeviceGetStreamPriorityRange(&plo, &phi);
    e = cudaStreamCreateWithPriority(&s->grp[g].stream, cudaStreamNonBlocking, plo);
    if (e == cudaSuccess && G > 1 && !getenv("SMPC_QP_NOPRIO")) e = cudaStreamCreateWithPriority(&s->grp[g].hi, cudaStreamNonBlocking, phi);
    for (int i = 0; i < RING && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&s->grp[g].ev[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->grp[g].ev_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->grp[g].evx, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->grp[g].body, cudaStreamNonBlocking);
  }
  if (e != cudaSuccess) { *err = e; qp_destroy(s); return nullptr; }
  double* p = s->block;
  s->q.it[0] = p; p += S * NIT;
  s->q.it[1] = p; p += S * NIT;
  s->q.res = p; p += S * NRES;
  s->q.stp = p; p += S * NSTP;
  s->q.pd = p; p += T * NPD * TL;
  qs_real* pr = reinterpret_cast<qs_real*>(p);
  s->q.rec = pr; pr += S * REC;
  s->q.st = pr; pr += S * NIT;
  s->q.st2 = pr; pr += S * NS2;
  s->q.sb = pr; pr += S * NSB;
  s->q.prod = pr;
  s->q.pi = s->pi;
  s->q.N = N;
  s->q.tile0 = 0;
  size_t mv_off = 0;
  for (int g = 0; g < G; ++g) {
    QpGroup& gr = s->grp[g];
    const int t0 = (int)((long long)s->T * g / G), t1 = (int)((long long)s->T * (g + 1) / G);
    const size_t so = (size_t)t0 * (N + 1) * TL;
    gr.T = t1 - t0;
    gr.q = s->q;
    gr.q.rec = s->q.rec + so * REC; gr.q.it[0] = s->q.it[0] + so * NIT; gr.q.it[1] = s->q.it[1] + so * NIT; gr.q.st = s->q.st + so * NIT; gr.q.st2 = s->q.st2 + so * NS2;
    gr.q.sb = s->q.sb + so * NSB; gr.q.prod = s->q.prod + so * NPROD; gr.q.res = s->q.res + so * NRES; gr.q.stp = s->q.stp + so * NSTP;
    gr.q.pd = s->q.pd + (size_t)t0 * NPD * TL; gr.q.pi = s->q.pi + (size_t)t0 * NPI * TL; gr.q.tile0 = t0;
    gr.counters = s->counters + ncnt * g;
    gr.h_counters = s->h_counters + 2 * RING * g;
    gr.mv_half = gr.T * TL / 2 + 1;
    gr.mv = s->mv + mv_off; mv_off += 2 * (size_t)gr.mv_half;
    gr.n_moves = s->n_moves + g;
    gr.redo_list = s->redo_list + (size_t)t0 * TL;
    gr.in_use = gr.T * TL;
    gr.kk_dev = s->kk_dev + g;
  }
  *err = cudaSuccess;
  return s;
}

void qp_destroy(QpSolver* s) {
  if (!s) return;
  for (int g = 0; g < MAX_GROUPS; ++g) {
    if (s->grp[g].stream) { cudaStreamSynchronize(s->grp[g].stream); cudaStreamDestroy(s->grp[g].stream); }
    if (s->grp[g].hi) { cudaStreamSynchronize(s->grp[g].hi); cudaStreamDestroy(s->grp[g].hi); }
    for (int i = 0; i < RING; ++i) if (s->grp[g].ev[i]) cudaEventDestroy(s->grp[g].ev[i]);
    if (s->grp[g].ev_done) cudaEventDestroy(s->grp[g].ev_done);
    if (s->grp[g].evx) cudaEventDestroy(s->grp[g].evx);
    if (s->grp[g].body) cudaStreamDestroy(s->grp[g].body);
  }
  if (s->ev_in) cudaEventDestroy(s->ev_in);
  if (s->block) cudaFree(s->block);
  if (s->pi) cudaFree(s->pi);
  if (s->counters) cudaFree(s->counters);
  if (s->kk_dev) cudaFree(s->kk_dev);
  if (s->h_counters) cudaFreeHost(s->h_counters);
  if (s->mv) cudaFree(s->mv);
  if (s->n_moves) cudaFree(s->n_moves);
  if (s->redo_list) cudaFree(s->redo_list);
  delete s;
}

void* qp_rec(QpSolver* s) { return const_cast<qs_real*>(s->q.rec); }
int qp_last_iterations(const QpSolver* s) { return s->last_iters; }
int qp_groups(const QpSolver* s) { return s->G; }
int qp_compactions(const QpSolver* s) { return s->n_compactions; }
void qp_set_profiling(QpSolver* s, bool on) { s->profile = on; }
bool qp_traced(const QpSolver* s) { return s->profile || s->trace_print; }
void qp_get_profile(const QpSolver* s, double* ms, int32_t* n, double* span_ms) {
  for (int i = 0; i < SMPC_PROF_N; ++i) { ms[i] = s->prof_ms[i]; n[i] = s->prof_n[i]; }
  *span_ms = s->prof_span_ms;
}

namespace {
static int prof_slot(const char* n) {
  static const char* names[SMPC_PROF_N] = {"qs_init_kernel", "qs_prep_kernel", "qs_ctl_kernel", "qs_ric1_kernel", "qs_step_kernel<0>", "qs_ric2_kernel",
                                           "qs_step_kernel<1>", "qs_red_kernel", "qs_compact" /* final + plan + move of a compaction */, "qs_step_kernel<2>", "qs_final_kernel",
                                           "qs_solo_kernel"};
  for (int i = 0; i < SMPC_PROF_N; ++i) if (names[i] && !strcmp(names[i], n)) return i;
  return 0;
}

// kernel launches of one tile group on its own stream
struct DeviceBackend {
  int64_t* launches;
  const smpc_problem_t* dP;
  QpSolver* s;
  QpGroup* g;
  const double* x0; const int32_t* r; const uint8_t* act;
  double *xt, *ut; int32_t *status, *qp_iter, *qp_status; double* qp_res;
  int kk_last = 0;
  int n_active_last = 1 << 30;  // problems still iterating after the newest control kernel the host has seen
  int n_redo_last = -1, n_redo_kk = -1;   // problems flagged for the centering direction in iteration n_redo_kk (the counters the host read last)
  bool red_done = false;        // the list form of the centering switch has already taken the step length: the next red(true) is a no-op
  cudaError_t err = cudaSuccess;
  bool on_hi = false;
  // solve captured into a CUDA graph (qs_graph_drive): no host reads; while the loop body is being captured, every kernel goes to the
  // body stream and takes its iteration from g->kk_dev, in the fixed forms of DESIGN §3.2
  bool graph = false;
  cudaStream_t in_body = nullptr;
  cudaGraphConditionalHandle cond = 0;
  const int* kd() const { return in_body ? g->kk_dev : nullptr; }
  bool trace_on() const { return s->profile || s->trace_print; }
  // stream for the next kernel; a change of stream is ordered after everything queued on the other one
  cudaStream_t st(bool hi) {
    if (in_body) return in_body;
    if (!g->hi) return g->stream;
    if (hi != on_hi) {
      cudaEventRecord(g->evx, on_hi ? g->hi : g->stream);
      cudaStreamWaitEvent(hi ? g->hi : g->stream, g->evx, 0);
      on_hi = hi;
    }
    return hi ? g->hi : g->stream;
  }
  // grids cover the tiles that may still hold an iterating problem (all of them until the first compaction)
  int tl() const { return g->tiles(); }
  int sp_grid() const { return (tl() * (s->N + 1) + SP_WARPS - 1) / SP_WARPS; }
  int sp_grid_all() const { return (g->T * (s->N + 1) + SP_WARPS - 1) / SP_WARPS; }
  void count(int n = 1) { *launches += n; }
  int gi() const { return (int)(g - s->grp); }
  void tr0(const char* name, cudaStream_t stm) {
    if (!trace_on()) return;
    TraceRec r{gi(), name, kk_last, nullptr, nullptr};
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, stm);
    s->trace.push_back(r);
  }
  void tr1(cudaStream_t stm) { if (trace_on()) cudaEventRecord(s->trace.back().b, stm); }
  void init() {
    g->in_use = g->T * TL;
    // (a captured solve may end up inside a conditional body, which takes kernel nodes only)
    if (graph) { launch_fill_i32(LaunchCtx{st(false), launches}, g->counters, 2 * (s->iter_max + 2), 0); }
    else cudaMemsetAsync(g->counters, 0, sizeof(int) * 2 * (s->iter_max + 2), st(false));
    { cudaStream_t stm_ = st(false); tr0("qs_init_kernel", stm_); qs_init_kernel<<<g->T, 32, 0, stm_>>>(g->q, s->B, x0, r, act); tr1(stm_); }
    count();
  }
  void prep(int kk) {
    {
      cudaStream_t stm_ = st(false);
      const int grid = (tl() * (s->N + 1) + PREP_WARPS - 1) / PREP_WARPS;
      tr0("qs_prep_kernel", stm_);
      if (kk == 0 && !in_body) qs_prep_kernel<true><<<grid, 32 * PREP_WARPS, PREP_SMEM, stm_>>>(dP, g->q, tl(), kk, nullptr);
      // the cooperative form stages whole (tile, stage) blocks, the thread-per-stage form only touches the lanes that still iterate:
      // measured break-even at about half of the slots in use active (full launch 0.57 ms against 1.02 ms).  In the deep tail (a handful
      // of tiles) throughput does not matter and the cooperative form has the shorter critical path (33 against 43 us)
      else if (s->coop_prep && (in_body || 2 * n_active_last >= g->in_use || n_active_last <= s->tail_max))
        qs_prep_coop_kernel<<<tl() * (s->N + 1), 32 * PC_WARPS, PC_SMEM, stm_>>>(dP, g->q, tl(), kk, kd());
      else qs_prep_kernel<false><<<grid, 32 * PREP_WARPS, PREP_SMEM, stm_>>>(dP, g->q, tl(), kk, kd());
      tr1(stm_);
    }
    count();
  }
  void ctl(int kk) {
    kk_last = kk;
    { cudaStream_t stm_ = st(false); tr0("qs_ctl_kernel", stm_); qs_ctl_kernel<<<tl(), 32, 0, stm_>>>(dP, g->q, kk, status, qp_iter, qp_status, qp_res, g->counters, kd()); tr1(stm_); }
    count();
  }
  void ric1() {
    {
      cudaStream_t stm_ = st(true);
      tr0("qs_ric1_kernel", stm_);
      if (!in_body && n_active_last <= s->tail_max && (s->tail_which & 1)) qs_ric1t_kernel<<<tl() * (32 / RT_WARPS), 32 * RT_WARPS, RT_SMEM, stm_>>>(dP, g->q);
      else if (s->split_ric1) qs_ric1x_kernel<<<tl(), 64, RIC1X_SMEM, stm_>>>(dP, g->q);
      else qs_ric1_kernel<<<tl(), 32, RIC1_SMEM, stm_>>>(dP, g->q);
      tr1(stm_);
    }
    count();
  }
  void ric2() {
    {
      cudaStream_t stm_ = st(true);
      tr0("qs_ric2_kernel", stm_);
      if (!in_body && n_active_last <= s->tail_max && (s->tail_which & 2)) qs_ric2t_kernel<<<tl() * (32 / RT_WARPS), 32 * RT_WARPS, RT_SMEM, stm_>>>(dP, g->q);
      else qs_ric2_kernel<<<tl(), 32, RIC2_SMEM, stm_>>>(dP, g->q);
      tr1(stm_);
    }
    count();
  }
  template <int MODE>
  void step_pass(cudaStream_t stm_, int kk, bool ring) {
    if (ring) qs_step_ring_kernel<MODE><<<sp_grid(), 32 * SP_WARPS, SR_SMEM, stm_>>>(dP, g->q, tl(), kk, kd());
    else qs_step_kernel<MODE><<<sp_grid(), 32 * SP_WARPS, 0, stm_>>>(dP, g->q, tl(), kk, kd());
  }
  void step(int kk, int mode) {
    if (mode == 0) { cudaStream_t stm_ = st(false); tr0("qs_step_kernel<0>", stm_); step_pass<0>(stm_, kk, s->ring_step); tr1(stm_); }
    else if (mode == 1) { cudaStream_t stm_ = st(false); tr0("qs_step_kernel<1>", stm_); step_pass<1>(stm_, kk, s->ring_step); tr1(stm_); }
    else {
      cudaStream_t stm_ = st(false);
      tr0("qs_step_kernel<2>", stm_);
      // (the host knows the number of flagged problems only when it has waited for the counters of THIS iteration: depth 0)
      const int lim = s->redo_list_max < 0 ? g->in_use / 8 : s->redo_list_max;
      if (!in_body && n_redo_kk == kk && n_redo_last > 0 && n_redo_last <= lim) {
        qs_redo_list_kernel<<<n_redo_last, RL_THREADS, 0, stm_>>>(dP, g->q, kk, g->redo_list, g->counters + 2 * kk + 1);
        red_done = true;
      } else step_pass<2>(stm_, kk, s->ring_step);
      tr1(stm_);
    }
    count();
  }
  // hand the rest of the solve (from the control phase of iteration kk on) to the solo kernel when few enough problems are left
  bool solo(int kk) {
    const int left = n_active_last < g->in_use ? n_active_last : g->in_use;
    if (s->solo_max <= 0 || left > s->solo_max || (kk > 0 && !s->solo_tail)) return false;
    kk_last = kk;
    cudaStream_t stm_ = st(false);
    tr0("qs_solo_kernel", stm_);
    qs_solo_kernel<<<tl() * TL, SOLO_THREADS, SOLO_SMEM, stm_>>>(dP, g->q, kk, status, qp_iter, qp_status, qp_res);
    tr1(stm_);
    count();
    return true;
  }
  // results of the problems that have finished and not been written yet; all slots of the group (empty ones are skipped)
  void final() { { cudaStream_t stm_ = st(false); tr0("qs_final_kernel", stm_); qs_final_kernel<<<sp_grid_all(), 32 * SP_WARPS, 0, stm_>>>(g->q, g->T, s->B, act, status, xt, ut); tr1(stm_); } count(); }
  void red(bool after) {
    if (after && red_done) { red_done = false; return; }
    { cudaStream_t stm_ = st(false); tr0("qs_red_kernel", stm_); qs_red_kernel<<<tl(), 32, 0, stm_>>>(dP, g->q, kk_last, after ? 1 : 0, g->counters, g->redo_list, kd()); tr1(stm_); }
    count();
  }
  // Compaction between iteration kk and kk + 1 (qp_split.cuh: qs_compact_*), decided on the newest active count the host has seen --
  // an upper bound of the current one, the counts never grow: when it has fallen to 85 % of the slots in use (and by at least a
  // tile), the problems still iterating are packed into the leading slots and every later launch covers only those tiles.
  void compact(int kk) {
    if (!s->compact || g->T < s->compact_min_tiles) return;
    const int na = n_active_last;
    if (na > g->in_use || g->in_use - na < TL || (double)na > s->compact_at * g->in_use) return;
    // in the tail (warp-per-problem sweeps, a handful of tiles) one compaction at its start is enough: a further one costs more
    // (three launches, ~0.1 ms) than the few tiles it would save
    if (na <= s->tail_max && g->in_use <= 2 * s->tail_max) return;
    cudaStream_t stm_ = st(false);
    tr0("qs_compact", stm_);
    const int tl_before = tl();
    qs_final_kernel<<<(tl_before * (s->N + 1) + SP_WARPS - 1) / SP_WARPS, 32 * SP_WARPS, 0, stm_>>>(g->q, tl_before, s->B, act, status, xt, ut);
    qs_compact_plan_kernel<<<1, CP_THREADS, 0, stm_>>>(g->q, tl_before, g->mv, g->mv_half, g->n_moves);
    const int grid_x = (g->in_use / 2) / 32 + 1;   // movers = min(active beyond the boundary, holes below it) <= half of the slots in use; 32 per CTA
    qs_compact_move_kernel<<<dim3(grid_x, s->N + 1), CM_THREADS, 0, stm_>>>(g->q, g->mv, g->mv_half, g->n_moves, kk);
    tr1(stm_);
    count(3);
    g->in_use = na;
    s->compacted = true;
    s->n_compactions += 1;
  }
  // Device-side loop (qs_graph_drive): a reset kernel, then a conditional WHILE node whose body graph is captured on g->body by one
  // call of body(*this); the node joins the capture of the group stream, and the kernels queued after loop() follow it
  template <class F>
  void loop(F body) {
    cudaStream_t stm_ = st(false);
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaGraph_t graph = nullptr;
    const cudaGraphNode_t* deps = nullptr;
    size_t n_deps = 0;
    cudaError_t e = cudaStreamGetCaptureInfo(stm_, &cs, nullptr, &graph, &deps, &n_deps);
    if (e == cudaSuccess && cs != cudaStreamCaptureStatusActive) e = cudaErrorStreamCaptureInvalidated;
    if (e == cudaSuccess) e = cudaGraphConditionalHandleCreate(&cond, graph, 1, cudaGraphCondAssignDefault);
    if (e == cudaSuccess) {
      qs_loop_reset_kernel<<<1, 1, 0, stm_>>>(g->kk_dev, cond);
      count();
      e = cudaStreamGetCaptureInfo(stm_, &cs, nullptr, &graph, &deps, &n_deps);
    }
    cudaGraphNodeParams np = {};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = cond;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t node = nullptr;
    if (e == cudaSuccess) e = cudaGraphAddNode(&node, graph, deps, n_deps, &np);
    // (a failure past this point leaves the capture holding a WHILE node with an empty body; the error is returned and the caller has to
    // discard the capture)
    if (e == cudaSuccess) e = cudaStreamUpdateCaptureDependencies(stm_, &node, 1, cudaStreamSetCaptureDependencies);
    if (e == cudaSuccess) e = cudaStreamBeginCaptureToGraph(g->body, np.conditional.phGraph_out[0], nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed);
    if (e != cudaSuccess) { err = e; return; }
    in_body = g->body;
    body(*this);
    in_body = nullptr;
    cudaGraph_t captured = nullptr;
    e = cudaStreamEndCapture(g->body, &captured);     // (the body graph belongs to the node)
    if (e != cudaSuccess && err == cudaSuccess) err = e;
  }
  void loop_step() {
    cudaStream_t stm_ = st(false);
    qs_loop_kernel<<<1, 1, 0, stm_>>>(g->counters, g->kk_dev, s->iter_max, cond);
    count();
  }
  void request_counters(int kk) {
    const int slot = kk % RING;
    cudaError_t e = cudaMemcpyAsync(g->h_counters + 2 * slot, g->counters + 2 * kk, 2 * sizeof(int), cudaMemcpyDeviceToHost, st(false));
    if (e == cudaSuccess) e = cudaEventRecord(g->ev[slot], st(false));
    if (e != cudaSuccess) err = e;
  }
  // counters of iteration kk: true when they have arrived (must: block until they have)
  bool wait_counters(int kk, bool must, int& na, int& nr) {
    const int slot = kk % RING;
    cudaError_t e = err;
    if (e == cudaSuccess) {
      if (must) e = cudaEventSynchronize(g->ev[slot]);
      else {
        e = cudaEventQuery(g->ev[slot]);
        if (e == cudaErrorNotReady) return false;
      }
    }
    if (e != cudaSuccess) { err = e; na = 0; nr = 0; return true; }     // stop iterating; the caller reports the error
    na = g->h_counters[2 * slot]; nr = g->h_counters[2 * slot + 1];
    n_active_last = na;
    n_redo_last = nr; n_redo_kk = kk;
    if (s->trace_print) fprintf(stderr, "QPCOUNT g=%d kk=%d active=%d redo=%d in_use=%d\n", gi(), kk, na, nr, g->in_use);
    return true;
  }
};
}  // namespace

cudaError_t launch_qp_solve(const LaunchCtx& c, const smpc_problem_t* dP, QpSolver* s, const double* x0, const int32_t* r, const uint8_t* act,
                            double* xt, double* ut, int32_t* status, int32_t* qp_iter, int32_t* qp_status, double* qp_res) {
  s->compacted = false; s->n_compactions = 0;
  // a solve captured into a CUDA graph runs its loop on the device (one tile group, no host-side timeline; api.cu refuses the rest
  // before anything is queued)
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaError_t e = cudaStreamIsCapturing(c.stream, &cs);
  if (e != cudaSuccess) return e;
  const bool graph = cs == cudaStreamCaptureStatusActive;
  if (graph && (s->G != 1 || s->profile || s->trace_print)) return cudaErrorNotSupported;
  // the group streams start after everything queued on the caller's stream (linearisation, input copies) ...
  e = cudaEventRecord(s->ev_in, c.stream);
  if (e != cudaSuccess) return e;
  DeviceBackend bk[MAX_GROUPS];
  for (int g = 0; g < s->G; ++g) {
    e = cudaStreamWaitEvent(s->grp[g].stream, s->ev_in, 0);
    if (e != cudaSuccess) return e;
    bk[g] = DeviceBackend{c.launches, dP, s, &s->grp[g], x0, r, act, xt, ut, status, qp_iter, qp_status, qp_res};
  }
  if (graph) {
    bk[0].graph = true;
    qs_graph_drive(bk[0]);
    if (bk[0].err != cudaSuccess) return bk[0].err;
    e = cudaEventRecord(s->grp[0].ev_done, bk[0].st(false));
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c.stream, s->grp[0].ev_done, 0);
    return e;
  }
  s->last_iters = qs_drive(bk, s->G, s->depth);
  if (s->profile || s->trace_print) {
    for (int g = 0; g < s->G; ++g) cudaStreamSynchronize(bk[g].st(false));
    if (!s->trace.empty()) {
      cudaEvent_t t0 = s->trace[0].a;
      for (int i = 0; i < SMPC_PROF_N; ++i) { s->prof_ms[i] = 0.0; s->prof_n[i] = 0; }
      float t_end = 0;
      for (auto& r : s->trace) {
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, t0, r.a); cudaEventElapsedTime(&b, t0, r.b);
        if (s->trace_print) fprintf(stderr, "QPTRACE g=%d kk=%d %-12s start=%9.3f end=%9.3f dur=%8.3f\n", r.g, r.kk, r.name, a, b, b - a);
        const int sl = prof_slot(r.name);
        s->prof_ms[sl] += b - a; s->prof_n[sl] += 1;
        t_end = b > t_end ? b : t_end;
      }
      s->prof_span_ms = t_end;
      for (auto& r : s->trace) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
      s->trace.clear();
    }
  }
  // ... and the caller's stream continues after the last kernel of every group
  for (int g = 0; g < s->G; ++g) {
    if (bk[g].err != cudaSuccess) return bk[g].err;
    e = cudaEventRecord(s->grp[g].ev_done, bk[g].st(false));
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c.stream, s->grp[g].ev_done, 0);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

void launch_rec_untile(const LaunchCtx& c, QpSolver* s, double* out) {
  const size_t n = (size_t)s->B * (s->N + 1) * REC;
  rec_untile_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c.stream>>>(s->B, s->N, s->q.rec, out);
  ++*c.launches;
}

void launch_dump_qp(const LaunchCtx& c, const smpc_problem_t* dP, QpSolver* s, double* dz, double* pi, double* lam, double* t) {
  const int n = s->B * (s->N + 1);
  dump_qp_kernel<<<(n + 127) / 128, 128, 0, c.stream>>>(dP, s->q, s->B, dz, pi, lam, t);
  ++*c.launches;
}

}  // inline namespace QS_FLAVOUR
}  // namespace smpc
