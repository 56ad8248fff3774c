// Stage-structured interior-point QP solve of one RTI iteration -- split formulation (v6).
//
// Replaces the HPIPM call inside AcadosOcpSolver.solve() (reference controller.py:158; options :97-110,208-209;
// algorithm: Frison & Diehl, HPIPM, IFAC 2020 -- Mehrotra predictor-corrector IPM, inequality rows condensed into
// the stage Hessian, backward Riccati factorisation / forward substitution) and the full-step update / status
// mapping acados' SQP_RTI performs around it (controller.py:161-167).
//
// Decomposition.  Only the Riccati recursion is sequential in the stage index k; the primal-dual update, the
// residuals, the condensation of the inequality rows, the recovery of (dlam, dt, dslack) and the step length are
// independent per (problem, stage).  One IPM iteration is therefore a short sequence of small kernels:
//   prep   (thread per (problem, stage))  update iterate, residuals, condensed stage matrix / gradient
//   ctl    (thread per problem)           reduce residual norms, convergence / failure logic, write result when done
//   ric1   (thread per problem)           backward factorisation + forward substitution of the affine direction
//   step0  (thread per (problem, stage))  affine (dlam, dt), step-length partials, dlam*dt products, corrector terms
//   ric2   (thread per problem)           sigma; vector-only backward + forward sweep of the corrector direction and, in the
//                                         same pass, of the pure-centering direction
//   step1  (thread per (problem, stage))  corrector (dlam, dt, dslack), step-length partials
//   red    (thread per problem)           step length; conditional predictor-corrector decision
//   step1 / red in mode 2                 the problems that asked for it switch to the centering direction
// Every lane owns a whole problem (or a whole stage of one): no shuffles, no barriers, no padding, 32 useful
// operations per instruction, and each kernel body is a few KB of code (the monolithic v5 kernel was bound by
// instruction fetch, profiles/r01_qp_v5_warp_per_problem.md).
//
// Layout.  Problems are grouped in tiles of TL = 32; every per-(problem, stage) array is stored
// [tile][stage][field][lane], every per-problem array [tile][field][lane]: lane l of a warp works on problem
// 32 tile + l and any field access of the warp is one coalesced 256-byte transaction, in the stage-parallel
// kernels (warp = one stage of a tile) and in the Riccati kernels (warp = one tile walking the stages) alike.
//
// QP variable order per stage: z = [du(5); dq(5); dv(5)].  The constant double-integrator A, B
// (env_model.py:63-71) are never stored: [B A]' P [B A] is formed in closed form from the 5x5 blocks of P.
// Rows per stage: box 0-9 (state j), torque 10-14, capsule 15-20, viability 21; slot = side * 22 + row,
// side 0 = lower, 1 = upper.  The viability row may be soft (one slack per side, L1 penalty).
//
// The functions are SMPC_HD so that tests/emu can run the very same source on the host against the oracle.
#pragma once
#include "dev_model.cuh"

// Storage flavour.  QS_REAL is the type of everything a solve STREAMS: stage records, search directions, condensed matrices and
// Riccati factors (rec, st, st2, sb, prod).  The iterate (z, pi, lam, t), the residual / step-length partials and the per-problem
// scalars are always fp64, and so is all arithmetic (values are widened on load, rounded on store).  The library holds both
// flavours: qp.cu is compiled once with QS_REAL = double (namespace smpc::f64, `precision = SMPC_PREC_F64`, bit-level parity
// with the oracle) and once with QS_REAL = float (qp_f32.cu, namespace smpc::f32, `precision = SMPC_PREC_F32`: 40 % less HBM
// traffic per interior-point iteration).  tests/emu compiles this header for the host in either flavour.
#ifndef QS_REAL
#define QS_REAL double
#define QS_FLAVOUR f64
#define QS_OTHER_FLAVOUR f32
#endif

namespace smpc {
inline namespace QS_FLAVOUR {
using qs_real = QS_REAL;

constexpr int TL = 32;             // problems per tile
constexpr int QNR = 22;            // two-sided rows per stage
SMPC_HD constexpr int tri(int i, int j) { return i * (i + 1) / 2 + j; }   // packed lower triangle, i >= j
SMPC_HD constexpr int trs(int i, int j) { return i >= j ? tri(i, j) : tri(j, i); }

// iterate block (also the layout of the step block)
enum { I_Z = 0, I_PIM = 15, I_LAM = 25, I_T = 69, I_SLK = 113, NIT = 120 };   // I_SLK: s_l s_u lam_sl lam_su t_sl t_su
// solver block of one stage: everything the Riccati sweeps read or write, ordered so that each sweep fetches one
// contiguous range:   ric1 backward reads [B_M, B_LP), writes [B_LP, B_V1);   ric1 forward reads [B_RB, B_WV);
// ric2 backward reads [B_GA, B_P) + [B_V1, NSB), writes B_LP, B_LP2;   ric2 forward reads [B_RB, B_V1)
//   M    condensed stage matrix H + reg + C' Gam C, packed lower triangle (prep)
//   GA   affine gradient res_g + C' gam (prep)          RB   dynamics residual of the link k -> k+1 (prep)
//   LP   l~ (5), p (10) of the current solve (ric1 / ric2)
//   T    elimination multipliers T[15][5], T[j][j] = 1/d_j (ric1)
//   WV   P_{k+1} res_b (ric1)                           P    Riccati matrix, packed 10x10 (ric1)
//   LP2  l~, p of the speculative centering solve (ric2)
//   V1   C'(dlam_aff dt_aff / t), V2 = C'(1 / t): corrector terms (step0)
enum { B_M = 0, B_GA = 120, B_RB = 135, B_LP = 145, B_T = 160, B_WV = 235, B_P = 245, B_LP2 = 300, B_V1 = 315, B_V2 = 330, NSB = 345 };
enum { H_M = B_M, H_GA = B_GA, H_RB = B_RB, F_LP = B_LP, F_T = B_T, F_WV = B_WV, F_P = B_P, F_LP2 = B_LP2, V_1 = B_V1, V_2 = B_V2, NHC = NSB, NFAC = NSB, NV = NSB };
enum { NS2 = 25 };                 // centering direction: dz (15), dpi (10), same field order as the step block
enum { NPROD = 46 };               // dlam_aff * dt_aff per slot (44) + the two slack slots
enum { R_NG = 0, R_NB = 1, R_ND = 2, R_NM = 3, R_MU = 4, R_CHK = 5, R_CNT = 6, NRES = 8 };
enum { S_ALPHA = 0, S_LIN = 1, S_QUAD = 2, NSTP = 4 };
// per-problem doubles
// D_RATIO, D_RESP: residual ratio max_i(res_i / tol_i) and residuals of the previous iterate (stall test of the fp32-storage flavour)
enum { D_X0 = 0, D_T0 = 10, D_MU = 65, D_MUAFF = 66, D_SIGMU = 67, D_ALPHA = 68, D_STEP = 69, D_RES = 70, D_RATIO = 74, D_RESP = 75, NPD = 80 };
// per-problem ints
// J_B: index of the problem this slot carries in the caller's arrays (-1: empty slot); J_FIN: its result (x_temp, u_temp) has been written
enum { J_ACT = 0, J_ITER = 1, J_QST = 2, J_REDO = 3, J_NC = 4, J_ITBUF = 5, J_R = 6, J_B = 7, J_FIN = 8, NPI = 9 };

struct QsBufs {
  const qs_real* rec;    // [T][N+1][REC][TL]   stage records (linearisation)
  double* it[2];         // [T][N+1][NIT][TL]   iterate, ping-pong (always fp64)
  qs_real* st;           // [T][N+1][NIT][TL]   step
  qs_real* st2;          // [T][N+1][NS2][TL]   pure-centering direction (dz, dpi) computed speculatively by ric2
  qs_real* sb;            // [T][N+1][NSB][TL]   solver block (condensed matrices, Riccati factors, corrector terms)
  qs_real* prod;         // [T][N+1][NPROD][TL]
  double* res;           // [T][N+1][NRES][TL]
  double* stp;           // [T][N+1][NSTP][TL]
  double* pd;            // [T][NPD][TL]
  int32_t* pi;           // [T][NPI][TL]
  int N;
  int tile0;             // first tile of this group in the batch (problem index b = 32 (tile0 + tile) + lane)
};

#define QF(p, f) (p)[(size_t)(f) * TL]

// Reciprocal of a positive, normal double.  Device: hardware seed (2^-23) + two Newton steps, i.e. within an ulp of the
// correctly rounded result and free of the special-case branch of an IEEE division.  Used for the pivots of the Riccati
// sweeps, which sit on the sequential path (measured: qs_ric1 0.46 -> 0.39 ms); the slot reciprocals of prep / step keep the
// IEEE division (the branch-free form made those kernels slower: more values live across the slots).
SMPC_HD double qs_rcp(double x) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
#else
  return 1.0 / x;
#endif
}

SMPC_HD size_t qs_blk(int tile, int N, int k, int nf, int lane) { return ((size_t)(tile * (N + 1) + k) * nf) * TL + lane; }
SMPC_HD size_t qs_pb(int tile, int nf, int lane) { return (size_t)tile * nf * TL + lane; }

struct StageFlags {
  bool tau, dist, nn, soft;
  double zpen;
};
SMPC_HD StageFlags qs_flags(const smpc_problem_t& P, int k) {
  StageFlags f;
  f.tau = k < P.N;
  f.dist = (k > 0) || P.stage0_collision_rows;
  f.nn = stage_has_nn(P, k);
  f.soft = f.nn && k == P.N && P.nn_terminal_soft;
  f.zpen = f.soft ? P.slack_penalty_e : -1.0;
  return f;
}

// box of dx_j at stage k (controller.py:49-55,144-145,300-306,530-536,701-707)
// xk: x_j of the guess at stage k (record field SMPC_REC_X + j)
SMPC_HD void qs_box_x(const smpc_problem_t& P, const QsBufs& q, int tile, int lane, int k, int j, double xk, double x0j, int rrec, double& lo, double& hi) {
  const int N = q.N;
  if (k == 0) { lo = x0j - xk; hi = lo; }
  else if (k == N) { lo = P.lbx_e[j] - xk; hi = P.ubx_e[j] - xk; }
  else if (P.controller == SMPC_CTRL_REAL_RECEDING) {
    if (k == rrec) { const double c = QF(q.rec + qs_blk(tile, N, k + 1, REC, lane), SMPC_REC_X + j); lo = c - 1e-3 - xk; hi = c + 1e-3 - xk; }
    else { lo = P.x_min[j] - xk; hi = P.x_max[j] - xk; }
  } else { lo = P.lbx[j] - xk; hi = P.ubx[j] - xk; }
}
SMPC_HD void qs_box(const smpc_problem_t& P, const QsBufs& q, int tile, int lane, int k, int j, double x0j, int rrec, double& lo, double& hi) {
  qs_box_x(P, q, tile, lane, k, j, QF(q.rec + qs_blk(tile, q.N, k, REC, lane), SMPC_REC_X + j), x0j, rrec, lo, hi);
}
// cold start of a box row: primal moved inside, slacks >= thr0
SMPC_HD double qs_zinit(double lo, double hi, double& tl, double& tu) {
  const double thr0 = 1e-1;
  double zc = 0.0;
  tl = zc - lo; tu = hi - zc;
  if (tl < thr0) {
    if (tu < thr0) { zc = 0.5 * (lo + hi); tl = thr0; tu = thr0; }
    else { tl = thr0; zc = lo + thr0; }
  } else if (tu < thr0) { tu = thr0; zc = hi - thr0; }
  return zc;
}

SMPC_HD double qs_rm(int mode, double lamt, double prod, double sigmu) {
  return mode == 0 ? lamt : (mode == 1 ? lamt + prod - sigmu : lamt - sigmu);
}

struct QsNorms {
  double ng, nb, nd, nm, mu, chk;
  int cnt;
};

// ================================================================================================================
// prep: (cold start | primal-dual update) + residuals + condensation.   thread = (problem, stage)
// ================================================================================================================
// jsm: lane-private on-chip scratch [PREP_SCRATCH][TL] (lane offset applied) that keeps the torque and capsule Jacobians
// of the stage between their three uses (row products, multiplier terms, condensation): each entry is read ~10 times.
enum { PREP_SCRATCH = 105 };
// A product that must stay a product.  With -fmad the compiler may contract  x*y + u*v  either way round, and it decides per
// kernel; the thread-per-stage and the cooperative form of prep must agree to the last bit (a problem's result must not depend on
// which form served it), so the few expressions with two candidate contractions are written with their rounding pinned.
// Slot reciprocals of prep (the same in both forms, so that they stay bit-identical): the branch-free reciprocal (measured 1 % of
// a solve faster than the IEEE division, which -DQS_SLOT_IEEE brings back).
#ifdef QS_SLOT_IEEE
#define QS_SRCP(x) (1.0 / (x))
#else
#define QS_SRCP(x) qs_rcp(x)
#endif
#ifdef __CUDA_ARCH__
#define QS_MUL(x, y) __dmul_rn((x), (y))
#else
#define QS_MUL(x, y) ((x) * (y))
#endif

template <bool FIRST>
SMPC_HD void qs_prep(const smpc_problem_t& P, const QsBufs& q, int tile, int lane, int k, int kk, double* jsm) {
  const int N = q.N;
  const int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  if (!QF(pi, J_ACT)) return;
  const double* pd = q.pd + qs_pb(tile, NPD, lane);
  constexpr bool first = FIRST;            // cold start (kk == 0) is its own instantiation: half the code, no runtime branches
  const double a = first ? 0.0 : QF(pd, D_STEP);
  const int rrec = QF(pi, J_R);
  const qs_real* rec = q.rec + qs_blk(tile, N, k, REC, lane);
  double* ito = q.it[kk & 1] + qs_blk(tile, N, k, NIT, lane);
  const double* iti = q.it[(kk & 1) ^ 1] + qs_blk(tile, N, k, NIT, lane);
  const qs_real* st = q.st + qs_blk(tile, N, k, NIT, lane);
  qs_real* hc = q.sb + qs_blk(tile, N, k, NHC, lane);
  const StageFlags F = qs_flags(P, k);
  const double lam_min = 1e-16, t_min = 1e-16, thr0 = 1e-1, mu0 = P.qp_mu0, reg = P.qp_reg_prim;
  const double dt = P.dt, a2 = 0.5 * P.dt * P.dt;
  QsNorms nr;
  nr.ng = nr.nb = nr.nd = nr.nm = nr.mu = nr.chk = 0.0; nr.cnt = 0;

  // ---- iterate of this stage ----
  double z[15], blo[10], bhi[10];
#pragma unroll
  for (int j = 0; j < 10; ++j) qs_box(P, q, tile, lane, k, j, QF(pd, D_X0 + j), rrec, blo[j], bhi[j]);
  if (first) {
#pragma unroll
    for (int i = 0; i < 5; ++i) z[i] = 0.0;
#pragma unroll
    for (int j = 0; j < 10; ++j) { double tl, tu; z[5 + j] = qs_zinit(blo[j], bhi[j], tl, tu); }
  } else {
#pragma unroll
    for (int i = 0; i < 15; ++i) z[i] = QF(iti, I_Z + i) + a * QF(st, I_Z + i);
  }
  if (k == N) {
#pragma unroll
    for (int i = 0; i < 5; ++i) z[i] = 0.0;
  }

  // ---- stationarity residual: H z + g + [B A]' pi_{k+1} - pi_k  (inequality multipliers are added row by row below) ----
  double rg[15], gd[15];
#pragma unroll
  for (int i = 0; i < 15; ++i) gd[i] = 0.0;
  {
    const double hu = QF(rec, SMPC_REC_HU), hq = QF(rec, SMPC_REC_HQ), hv = QF(rec, SMPC_REC_HV);
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      rg[i] = (k == N) ? 0.0 : hu * z[i] + QF(rec, SMPC_REC_G + i);
      double s = QF(rec, SMPC_REC_G + 5 + i) + hq * z[5 + i];
#pragma unroll
      for (int j = 0; j < 5; ++j) s += QF(rec, SMPC_REC_HQQ + trs(i, j)) * z[5 + j];
      rg[5 + i] = s;
      rg[10 + i] = QF(rec, SMPC_REC_G + 10 + i) + hv * z[10 + i];
    }
  }
  // multipliers of the dynamics: pi_k (link k-1 -> k, stored with stage k), pi_{k+1}
  double pimv[10];
#pragma unroll
  for (int j = 0; j < 10; ++j) {
    pimv[j] = (first || k == 0) ? 0.0 : QF(iti, I_PIM + j) + a * QF(st, I_PIM + j);
    rg[5 + j] -= pimv[j];
  }
  if (k < N) {
    const double* itn = q.it[(kk & 1) ^ 1] + qs_blk(tile, N, k + 1, NIT, lane);
    const qs_real* stn = q.st + qs_blk(tile, N, k + 1, NIT, lane);
    double rb[10];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      rb[j] = z[5 + j] + dt * z[10 + j] + a2 * z[j] + QF(rec, SMPC_REC_B + j);
      rb[5 + j] = z[10 + j] + dt * z[j] + QF(rec, SMPC_REC_B + 5 + j);
    }
    if (first) {
#pragma unroll
      for (int j = 0; j < 10; ++j) {
        double lo, hi, tl, tu;
        qs_box(P, q, tile, lane, k + 1, j, 0.0, rrec, lo, hi);
        rb[j] -= qs_zinit(lo, hi, tl, tu);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const double pq = QF(itn, I_PIM + j) + a * QF(stn, I_PIM + j);
        const double pv = QF(itn, I_PIM + 5 + j) + a * QF(stn, I_PIM + 5 + j);
        if (k < N) { rg[j] += fma(a2, pq, QS_MUL(dt, pv)); }
        rg[5 + j] += pq;
        rg[10 + j] += dt * pq + pv;
        rb[j] -= QF(itn, I_Z + 5 + j) + a * QF(stn, I_Z + 5 + j);
        rb[5 + j] -= QF(itn, I_Z + 10 + j) + a * QF(stn, I_Z + 10 + j);
      }
    }
#pragma unroll
    for (int j = 0; j < 10; ++j) { QF(hc, H_RB + j) = rb[j]; nr.nb = fmax(nr.nb, fabs(rb[j])); nr.chk += rb[j]; }
  }
  // (stores of this phase come after all of its loads, see the note on the row phases below)
#pragma unroll
  for (int i = 0; i < 15; ++i) QF(ito, I_Z + i) = z[i];
#pragma unroll
  for (int j = 0; j < 10; ++j) QF(ito, I_PIM + j) = pimv[j];

  // ---- rows: (lam, t) update or cold start, residuals, condensation terms ----
  // Loads and stores are kept in separate phases (all row products and all updated (lam, t) of a row group first, then
  // the stores): the compiler may not move a load above a store it cannot prove disjoint, and one load round trip per
  // slot would serialise the thread on memory latency.
  auto upd = [&](int slot, double tinit, double& lam, double& t) {
    if (first) { t = tinit; lam = mu0 / t; }
    else {
      lam = fmax(QF(iti, I_LAM + slot) + a * QF(st, I_LAM + slot), lam_min);
      t = fmax(QF(iti, I_T + slot) + a * QF(st, I_T + slot), t_min);
    }
  };
  // one side of a row; returns G = lam/t and c = (lam t - lam r)/t  (mode-0 right-hand side)
  // mu is summed in four partial sums -- box rows 0-3, box rows 4-9, torque rows, capsule + viability rows (+ slacks) -- and the
  // partial sums in that order: the row groups of the four warps of qs_prep_coop, so that both forms round alike
  double mup[4] = {0.0, 0.0, 0.0, 0.0};
  auto side = [&](int slot, double sgn, double az, double bnd, double slack, double lam, double t, double& G, double& c) {
    QF(ito, I_LAM + slot) = lam; QF(ito, I_T + slot) = t;
    const double r = t - (sgn * (az - bnd) + slack);
    const double rm = QS_MUL(lam, t);                      // (QS_MUL: see the note at its definition)
    const double it_ = QS_SRCP(t);
    G = QS_MUL(lam, it_);
    c = QS_MUL(fma(-lam, r, rm), it_);
    mup[slot % QNR < 4 ? 0 : (slot % QNR < 10 ? 1 : (slot % QNR < 15 ? 2 : 3))] += rm;
    nr.chk += rm + r; nr.nm = fmax(nr.nm, fabs(rm)); nr.nd = fmax(nr.nd, fabs(r)); nr.cnt += 1;
  };
  // row products and bounds of the general rows (loads only)
  double azg[12], glo[12], ghi[12];
#pragma unroll
  for (int r = 0; r < 12; ++r) { azg[r] = 0.0; glo[r] = 0.0; ghi[r] = 0.0; }
  if (F.tau) {
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      double az = 0.0;
#pragma unroll
      for (int c = 0; c < 15; ++c) { const double jv = QF(rec, SMPC_REC_JTAU + r * 15 + c); QF(jsm, r * 15 + c) = jv; az += jv * z[c]; }
      const double v = QF(rec, SMPC_REC_TAU + r);
      azg[r] = az; glo[r] = P.tau_min[r] - v; ghi[r] = P.tau_max[r] - v;
    }
  }
  if (F.dist) {
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      double az = 0.0;
#pragma unroll
      for (int c = 0; c < 5; ++c) { const double jv = QF(rec, SMPC_REC_JDIST + p * 5 + c); QF(jsm, 75 + p * 5 + c) = jv; az += jv * z[5 + c]; }
      const double v = QF(rec, SMPC_REC_DIST + p);
      azg[5 + p] = az; glo[5 + p] = P.pair_lo_ocp[p] - v; ghi[5 + p] = P.pair_hi - v;
    }
  }
  if (F.nn) {
    double az = 0.0;
#pragma unroll
    for (int c = 0; c < 10; ++c) az += QF(rec, SMPC_REC_JNN + c) * z[5 + c];
    const double v = QF(rec, SMPC_REC_NN);
    azg[11] = az; glo[11] = 0.0 - v; ghi[11] = 1e6 - v;
  }
  double Gb[10], Gg[12];
  // box rows
  {
    double bl[20], bt[20];
#pragma unroll
    for (int j = 0; j < 10; ++j) {
      double tl = 0.0, tu = 0.0;
      if (first) qs_zinit(blo[j], bhi[j], tl, tu);
      upd(j, tl, bl[j], bt[j]);
      upd(QNR + j, tu, bl[10 + j], bt[10 + j]);
    }
#pragma unroll
    for (int j = 0; j < 10; ++j) {
      double Gl, Gu, cl, cu;
      side(j, 1.0, z[5 + j], blo[j], 0.0, bl[j], bt[j], Gl, cl);
      side(QNR + j, -1.0, z[5 + j], bhi[j], 0.0, bl[10 + j], bt[10 + j], Gu, cu);
      Gb[j] = Gl + Gu;
      rg[5 + j] += bl[10 + j] - bl[j];
      gd[5 + j] += cl - cu;
    }
  }
  // general rows: updated (lam, t) of every slot, slack triplets of the soft row
  double gl[24], gt[24];
#pragma unroll
  for (int r = 0; r < 12; ++r) {
    const bool pres = r < 5 ? F.tau : (r < 11 ? F.dist : F.nn);
    gl[r] = gt[r] = gl[12 + r] = gt[12 + r] = 0.0;
    if (pres) {
      upd(10 + r, fmax(thr0, azg[r] - glo[r]), gl[r], gt[r]);
      upd(QNR + 10 + r, fmax(thr0, ghi[r] - azg[r]), gl[12 + r], gt[12 + r]);
    }
  }
  double sl[2] = {0.0, 0.0}, ls[2] = {0.0, 0.0}, ts[2] = {0.0, 0.0};
  if (F.soft) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (first) { sl[h] = thr0; ls[h] = mu0 / thr0; ts[h] = thr0; }
      else {
        sl[h] = QF(iti, I_SLK + h) + a * QF(st, I_SLK + h);
        ls[h] = fmax(QF(iti, I_SLK + 2 + h) + a * QF(st, I_SLK + 2 + h), lam_min);
        ts[h] = fmax(QF(iti, I_SLK + 4 + h) + a * QF(st, I_SLK + 4 + h), t_min);
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 12; ++r) Gg[r] = 0.0;
  if (F.tau) {
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      double Gl, Gu, cl, cu;
      side(10 + r, 1.0, azg[r], glo[r], 0.0, gl[r], gt[r], Gl, cl);
      side(QNR + 10 + r, -1.0, azg[r], ghi[r], 0.0, gl[12 + r], gt[12 + r], Gu, cu);
      Gg[r] = Gl + Gu;
      const double nu = gl[12 + r] - gl[r], gam = cl - cu;
#pragma unroll
      for (int c = 0; c < 15; ++c) { const double jv = QF(jsm, r * 15 + c); rg[c] += jv * nu; gd[c] += jv * gam; }
    }
  }
  if (F.dist) {
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      const int r = 5 + p;
      double Gl, Gu, cl, cu;
      side(10 + r, 1.0, azg[r], glo[r], 0.0, gl[r], gt[r], Gl, cl);
      side(QNR + 10 + r, -1.0, azg[r], ghi[r], 0.0, gl[12 + r], gt[12 + r], Gu, cu);
      Gg[r] = Gl + Gu;
      const double nu = gl[12 + r] - gl[r], gam = cl - cu;
#pragma unroll
      for (int c = 0; c < 5; ++c) { const double jv = QF(jsm, 75 + p * 5 + c); rg[5 + c] += jv * nu; gd[5 + c] += jv * gam; }
    }
  }
  // viability row (may be soft)
  if (F.nn) {
#pragma unroll
    for (int h = 0; h < 2; ++h) { QF(ito, I_SLK + h) = sl[h]; QF(ito, I_SLK + 2 + h) = ls[h]; QF(ito, I_SLK + 4 + h) = ts[h]; }
    const double ll = gl[11], lu = gl[23];
    double Gl, Gu, cl, cu;
    side(21, 1.0, azg[11], glo[11], sl[0], gl[11], gt[11], Gl, cl);
    side(QNR + 21, -1.0, azg[11], ghi[11], sl[1], gl[23], gt[23], Gu, cu);
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
        mup[3] += rms; nr.chk += rms + rsl + rgs;
        nr.nm = fmax(nr.nm, fabs(rms)); nr.nd = fmax(nr.nd, fabs(rsl)); nr.ng = fmax(nr.ng, fabs(rgs));
        nr.cnt += 1;
      }
      Gl = G2[0]; Gu = G2[1]; cl = c2[0]; cu = c2[1];
    }
    Gg[11] = Gl + Gu;
    const double nu = lu - ll, gam = cl - cu;
#pragma unroll
    for (int c = 0; c < 10; ++c) { const double jv = QF(rec, SMPC_REC_JNN + c); rg[5 + c] += jv * nu; gd[5 + c] += jv * gam; }
  }
  if (k == N) {
#pragma unroll
    for (int i = 0; i < 5; ++i) { rg[i] = 0.0; gd[i] = 0.0; }
  }
#pragma unroll
  for (int i = 0; i < 15; ++i) { nr.ng = fmax(nr.ng, fabs(rg[i])); nr.chk += rg[i]; QF(hc, H_GA + i) = rg[i] + gd[i]; }

  // ---- condensed stage matrix  H + reg + C' Gam C  (packed lower triangle) ----
  {
    const double hu = (k == N) ? 1.0 : QF(rec, SMPC_REC_HU) + reg;
    const double hq = QF(rec, SMPC_REC_HQ) + reg, hv = QF(rec, SMPC_REC_HV) + reg;
#pragma unroll
    for (int i = 0; i < 15; ++i) {
      double acc[15];
#pragma unroll
      for (int c = 0; c <= i; ++c) {
        double v = 0.0;
        if (c == i) v = i < 5 ? hu : ((i < 10 ? hq : hv) + Gb[i >= 5 ? i - 5 : 0]);
        if (i >= 5 && i < 10 && c >= 5) v += QF(rec, SMPC_REC_HQQ + tri(i - 5, c - 5));
        acc[c] = v;
      }
      if (F.tau) {
#pragma unroll
        for (int r = 0; r < 5; ++r) {
          const double w = Gg[r] * QF(jsm, r * 15 + i);
#pragma unroll
          for (int c = 0; c <= i; ++c) acc[c] += w * QF(jsm, r * 15 + c);
        }
      }
      if (F.dist && i >= 5 && i < 10) {
#pragma unroll
        for (int p = 0; p < 6; ++p) {
          const double w = Gg[5 + p] * QF(jsm, 75 + p * 5 + i - 5);
#pragma unroll
          for (int c = 5; c <= i; ++c) acc[c] += w * QF(jsm, 75 + p * 5 + c - 5);
        }
      }
      if (F.nn && i >= 5) {
        const double w = Gg[11] * QF(rec, SMPC_REC_JNN + i - 5);
#pragma unroll
        for (int c = 5; c <= i; ++c) acc[c] += w * QF(rec, SMPC_REC_JNN + c - 5);
      }
#pragma unroll
      for (int c = 0; c <= i; ++c) QF(hc, H_M + tri(i, c)) = acc[c];
    }
  }
  double* res = q.res + qs_blk(tile, N, k, NRES, lane);
  QF(res, R_NG) = nr.ng; QF(res, R_NB) = nr.nb; QF(res, R_ND) = nr.nd; QF(res, R_NM) = nr.nm;
  QF(res, R_MU) = ((mup[0] + mup[1]) + mup[2]) + mup[3]; QF(res, R_CHK) = nr.chk; QF(res, R_CNT) = (double)nr.cnt;
}

// ================================================================================================================
// ctl: residual norms of the new iterate, exit tests (same control flow as the oracle's QpIpm::solve), result.
// thread = problem.  Returns true when the problem stays active.
// ================================================================================================================
// CH: stages whose residuals are loaded together (the per-tile kernel uses 16: qs_ctl 1.05 -> 0.69 ms per cfg[1] solve; 0 = plain loop: the solo
// kernel, whose thread 0 runs this between the phases of a 255-register kernel, and the host emulation).  Same accumulation order either way.
template <int CH = 0>
SMPC_HD bool qs_ctl(const smpc_problem_t& P, const QsBufs& q, int tile, int lane, int kk_in, int32_t* status, int32_t* qp_iter,
                    int32_t* qp_status, double* qp_res) {
  const int N = q.N;
  int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  if (!QF(pi, J_ACT)) return false;
  double* pd = q.pd + qs_pb(tile, NPD, lane);
  int kk = kk_in;
  double ng = 0.0, nb = 0.0, nd = 0.0, nm = 0.0, mu = 0.0, chk = 0.0, cnt = 0.0;
  if constexpr (CH == 0) {
#pragma unroll 8
    for (int k = 0; k <= N; ++k) {
      const double* res = q.res + qs_blk(tile, N, k, NRES, lane);
      ng = fmax(ng, QF(res, R_NG)); nb = fmax(nb, QF(res, R_NB)); nd = fmax(nd, QF(res, R_ND)); nm = fmax(nm, QF(res, R_NM));
      mu += QF(res, R_MU); chk += QF(res, R_CHK); cnt += QF(res, R_CNT);
    }
  } else {
    // One warp per tile and a loop over the stages: the launch lasts as long as the load round trips of one thread, so the loop runs in
    // chunks of CH stages -- all loads of a chunk first (112 in flight for CH = 16), then the accumulation in stage order.
    constexpr int C = CH > 0 ? CH : 1;
    for (int k0 = 0; k0 <= N; k0 += C) {
      double v[C][7];
#pragma unroll
      for (int j = 0; j < C; ++j) {
        if (k0 + j <= N) {
          const double* res = q.res + qs_blk(tile, N, k0 + j, NRES, lane);
          v[j][0] = QF(res, R_NG); v[j][1] = QF(res, R_NB); v[j][2] = QF(res, R_ND); v[j][3] = QF(res, R_NM);
          v[j][4] = QF(res, R_MU); v[j][5] = QF(res, R_CHK); v[j][6] = QF(res, R_CNT);
        }
      }
#pragma unroll
      for (int j = 0; j < C; ++j) {
        if (k0 + j <= N) {
          ng = fmax(ng, v[j][0]); nb = fmax(nb, v[j][1]); nd = fmax(nd, v[j][2]); nm = fmax(nm, v[j][3]);
          mu += v[j][4]; chk += v[j][5]; cnt += v[j][6];
        }
      }
    }
  }
  if (kk == 0) QF(pi, J_NC) = (int)(cnt + 0.5);
  const int nc = QF(pi, J_NC);
  double r0 = (chk != chk) ? chk : ng;
  mu = mu / nc;
  QF(pd, D_RES + 0) = r0; QF(pd, D_RES + 1) = nb; QF(pd, D_RES + 2) = nd; QF(pd, D_RES + 3) = nm; QF(pd, D_MU) = mu;
  const bool nan = (r0 != r0) || (nb != nb) || (nd != nd) || (nm != nm);
  const bool unconv = (r0 > P.qp_tol_stat) || (nb > P.qp_tol_eq) || (nd > P.qp_tol_ineq) || (nm > P.qp_tol_comp);
  bool done = false;
  if (nan && kk > 0) done = true;
  else if (!unconv && !nan) done = true;
  else if (kk >= P.qp_iter_max) done = true;
  else if (!(QF(pd, D_ALPHA) > P.qp_alpha_min)) done = true;
  // fp32-storage flavour only.  The stored search direction carries a relative rounding of 6e-8 that the condensation amplifies by
  // lam / t, so the residuals of an iterate bottom out (1e-5 .. 1e-4 on this path) and GROW again if the iteration goes on.  A
  // solve that has come within qp_maxiter_accept x its tolerances and whose new iterate is worse than the previous one ends on
  // the previous iterate (still intact in the other ping-pong buffer) and reports it like an exit at the iteration limit.
  bool stalled = false;
  if (sizeof(qs_real) == 4) {
    const double ratio = nan ? 1e300 : fmax(fmax(r0 / P.qp_tol_stat, nb / P.qp_tol_eq), fmax(nd / P.qp_tol_ineq, nm / P.qp_tol_comp));
    const double prev = kk == 0 ? 1e300 : QF(pd, D_RATIO);
    const double F = P.qp_maxiter_accept > 0.0 ? P.qp_maxiter_accept : 1e3;
    if (kk >= 2 && (unconv || nan) && prev <= F && ratio > prev) { stalled = true; done = true; }
    if (!stalled) {
      QF(pd, D_RATIO) = ratio;
      QF(pd, D_RESP + 0) = r0; QF(pd, D_RESP + 1) = nb; QF(pd, D_RESP + 2) = nd; QF(pd, D_RESP + 3) = nm; QF(pd, D_RESP + 4) = mu;
    }
  }
  if (!done) return true;
  int qst;
  if (stalled) {
    qst = 1;
    r0 = QF(pd, D_RESP + 0); nb = QF(pd, D_RESP + 1); nd = QF(pd, D_RESP + 2); nm = QF(pd, D_RESP + 3); mu = QF(pd, D_RESP + 4);
    QF(pd, D_RES + 0) = r0; QF(pd, D_RES + 1) = nb; QF(pd, D_RES + 2) = nd; QF(pd, D_RES + 3) = nm;
    kk -= 1;                                               // the iterate that is reported
  } else if (nan) qst = 3; else if (!unconv) qst = 0; else if (kk >= P.qp_iter_max) qst = 1; else qst = 2;
  QF(pi, J_ACT) = 0; QF(pi, J_ITER) = kk; QF(pi, J_QST) = qst; QF(pi, J_ITBUF) = kk & 1;
  // status mapping of acados SQP_RTI: QP success / max-iter -> step taken (qs_final writes it), else QP failure.  A max-iter exit
  // counts as solved only when its iterate is within qp_maxiter_accept x the tolerances (smpc_problem_t::qp_maxiter_accept: an
  // infeasible QP ends at max-iter or at the minimum step length depending on rounding, with residuals many orders above)
  const int b = QF(pi, J_B);
  const double F = P.qp_maxiter_accept;
  const bool sane = !(F > 0.0) || (r0 <= F * P.qp_tol_stat && nb <= F * P.qp_tol_eq && nd <= F * P.qp_tol_ineq && nm <= F * P.qp_tol_comp);
  status[b] = (qst == 0 || (qst == 1 && sane)) ? 0 : 4;
  qp_iter[b] = kk;
  qp_status[b] = qst;
  for (int c = 0; c < 4; ++c) qp_res[(size_t)b * 5 + c] = QF(pd, D_RES + c);
  qp_res[(size_t)b * 5 + 4] = mu;
  return false;
}

// final: full step x_temp = x_guess + dx, u_temp = u_guess + du of one stage of a problem that took part in this solve and has
// finished but not been written yet (zero step after a QP failure; a NaN in an accepted step turns the status into acados' 1).
// Called once at the end of a solve and, when the solve compacts its slots, before every compaction (the slot of a finished
// problem may be reused then).   thread = (slot, stage)
// returns the problem index when this stage found a NaN in an accepted step (the caller raises status[b] to 1), else -1
SMPC_HD int qs_final(const QsBufs& q, int tile, int lane, int k, const uint8_t* act, int B, const int32_t* status, double* xt, double* ut) {
  const int N = q.N;
  const int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  const int b = QF(pi, J_B);
  if (b < 0 || b >= B || (act && !act[b])) return -1;
  if (QF(pi, J_ACT) || QF(pi, J_FIN)) return -1;
  const bool ok = status[b] != 4;
  const double* it = q.it[QF(pi, J_ITBUF)] + qs_blk(tile, N, k, NIT, lane);
  const qs_real* rec = q.rec + qs_blk(tile, N, k, REC, lane);
  bool znan = false;
  if (k < N) {
    double* utb = ut + ((size_t)b * N + k) * NU;
#pragma unroll
    for (int j = 0; j < NU; ++j) { const double z = ok ? QF(it, I_Z + j) : 0.0; znan |= (z != z); utb[j] = QF(rec, SMPC_REC_U + j) + z; }
  }
  double* xtb = xt + ((size_t)b * (N + 1) + k) * NX;
#pragma unroll
  for (int j = 0; j < NX; ++j) { const double z = ok ? QF(it, I_Z + NU + j) : 0.0; znan |= (z != z); xtb[j] = QF(rec, SMPC_REC_X + j) + z; }
  return znan ? b : -1;
}

// ================================================================================================================
// Compaction of the slots of a tile group.  The stage-parallel kernels stream whole tiles: a tile with one problem still
// iterating costs as much as a full one, and the iteration counts of the problems of a batch spread over a factor of two.
// Between two iterations the problems still iterating are therefore packed into the leading slots: with n active problems,
// the active ones in slots >= n (in slot order) move into the inactive slots < n (in slot order); nobody else moves, sources
// and destinations are disjoint, and every kernel then only walks the first ceil(n / 32) tiles.  A move copies bits (stage
// records, current iterate, step, per-problem scalars), so results do not depend on it.  The results of the finished
// problems are written by qs_final before their slots are reused.
// ================================================================================================================
// plan for one group of T tiles (serial form: tests/emu; the device builds the same plan with a block-wide scan, qp.cu).
// mv: [2][T * TL / 2] source and destination slots; returns the number of moves and marks the finished slots as written.
SMPC_HD int qs_compact_plan(const QsBufs& q, int T, int32_t* mv, int* n_active_out) {
  const int S = T * TL, half = S / 2;
  int n = 0;
  for (int s = 0; s < S; ++s) {
    int32_t* pi = q.pi + qs_pb(s / TL, NPI, s % TL);
    if (QF(pi, J_ACT)) ++n; else QF(pi, J_FIN) = 1;
  }
  int nm = 0, hole = 0;
  for (int s = n; s < S; ++s) {
    if (!QF(q.pi + qs_pb(s / TL, NPI, s % TL), J_ACT)) continue;
    while (QF(q.pi + qs_pb(hole / TL, NPI, hole % TL), J_ACT)) ++hole;
    mv[nm] = s; mv[half + nm] = hole; ++nm; ++hole;
  }
  if (n_active_out) *n_active_out = n;
  return nm;
}
// one field of one stage of one move (thread = (move, stage, field) on the device): what prep of the next iteration reads
// -- stage record, iterate of iteration kk, step
enum { CMP_FIELDS = REC + 2 * NIT };
SMPC_HD void qs_compact_move_field(const QsBufs& q, int src, int dst, int k, int kk, int f) {
  const int N = q.N;
  const int ts = src / TL, ls = src % TL, td = dst / TL, ld = dst % TL;
  if (f < REC) { qs_real* r = const_cast<qs_real*>(q.rec); QF(r + qs_blk(td, N, k, REC, ld), f) = QF(q.rec + qs_blk(ts, N, k, REC, ls), f); }
  else if (f < REC + NIT) { double* it = q.it[kk & 1]; QF(it + qs_blk(td, N, k, NIT, ld), f - REC) = QF(it + qs_blk(ts, N, k, NIT, ls), f - REC); }
  else QF(q.st + qs_blk(td, N, k, NIT, ld), f - REC - NIT) = QF(q.st + qs_blk(ts, N, k, NIT, ls), f - REC - NIT);
}
// per-problem scalars of one move; the source slot becomes empty
SMPC_HD void qs_compact_move_scalars(const QsBufs& q, int src, int dst) {
  int32_t* ps = q.pi + qs_pb(src / TL, NPI, src % TL);
  int32_t* pdst = q.pi + qs_pb(dst / TL, NPI, dst % TL);
  for (int f = 0; f < NPI; ++f) QF(pdst, f) = QF(ps, f);
  double* ds = q.pd + qs_pb(src / TL, NPD, src % TL);
  double* dd = q.pd + qs_pb(dst / TL, NPD, dst % TL);
  for (int f = 0; f < NPD; ++f) QF(dd, f) = QF(ds, f);
  QF(ps, J_ACT) = 0; QF(ps, J_FIN) = 1; QF(ps, J_B) = -1;
}

// ================================================================================================================
// Riccati sweeps.   thread = problem, walking the stages.
// Y = [B A]' P [B A] entry (i, c) of the 15x15 matrix, from the packed 10x10 P (rows/cols: q 0-4, v 5-9).
// ================================================================================================================
template <class PF>
SMPC_HD double qs_y(int i, int c, double dt, double a2, PF Pn) {
  const int gi = i / 5, gc = c / 5, ii = i % 5, ic = c % 5;
  // coefficient of q+ / v+ for the variable groups u, q, v
  const double aqi = gi == 0 ? a2 : (gi == 1 ? 1.0 : dt), avi = gi == 0 ? dt : (gi == 1 ? 0.0 : 1.0);
  const double aqc = gc == 0 ? a2 : (gc == 1 ? 1.0 : dt), avc = gc == 0 ? dt : (gc == 1 ? 0.0 : 1.0);
  double y = 0.0;
  y += (aqi * aqc) * Pn(trs(ii, ic));               // Pqq
  if (gc != 1) y += (aqi * avc) * Pn(tri(5 + ic, ii));   // Pqv[ii][ic] = P[ii][5+ic]
  if (gi != 1) y += (avi * aqc) * Pn(tri(5 + ii, ic));   // Pvq[ii][ic] = P[5+ii][ic]
  if (gi != 1 && gc != 1) y += (avi * avc) * Pn(trs(5 + ii, 5 + ic));
  return y;
}

// The sweeps are written against a small warp policy W (lane id, warp barrier, staged copies of a contiguous field
// range of a stage block into on-chip memory one stage ahead of its use): TMA bulk copies + mbarriers on the device
// (qp.cu), memcpy in tests/emu.  w.buf(b) is staging buffer b with this lane's offset applied, field f at [f * TL].
enum { RIC1_STAGE_FIELDS = B_LP - B_M, RIC2_STAGE_FIELDS = B_V1 - B_RB };   // largest range each kernel stages (145, 165)

// ric1: backward factorisation with the affine gradient, stage-0 solve, forward substitution of the affine direction.
// psm: on-chip scratch for the packed P matrix + p of the running stage, [65][TL] doubles (lane offset applied).
template <class W>
SMPC_HD void qs_ric1(const smpc_problem_t& P, const QsBufs& q, int tile, W& w, double* psm) {
  const int N = q.N, lane = w.lane();
  const int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  const bool on = QF(pi, J_ACT) != 0;
  if (!w.any(on)) return;
  double* pd = q.pd + qs_pb(tile, NPD, lane);
  const double dt = P.dt, a2 = 0.5 * P.dt * P.dt;
  const qs_real* gsb = q.sb + qs_blk(tile, N, 0, NSB, 0);       // stage blocks of this tile (no lane offset)
  const size_t sstride = (size_t)NSB * TL;
  double dx[10];
  // staging: with two buffers stage k - 1 is fetched while stage k is processed; with one buffer (more warps per SM)
  // the fetch of stage k - 1 is issued once every lane is done with stage k
  const int nb1 = w.nbuf() - 1;
  w.fetch_begin(N & nb1, B_LP - B_M);
  w.fetch(N & nb1, 0, gsb + (size_t)N * sstride, B_M, B_LP - B_M);
  for (int k = N; k >= 0; --k) {
    w.sync();                                                    // every lane is done with the buffer of stage k + 1
    if (nb1 && k > 0) { w.fetch_begin((k - 1) & 1, B_LP - B_M); w.fetch((k - 1) & 1, 0, gsb + (size_t)(k - 1) * sstride, B_M, B_LP - B_M); }
    if (!nb1 && k < N) { w.fetch_begin(0, B_LP - B_M); w.fetch(0, 0, gsb + (size_t)k * sstride, B_M, B_LP - B_M); }
    if (!nb1 && k > 0) w.prefetch(gsb + (size_t)(k - 1) * sstride, B_M, B_LP - B_M);      // next stage on its way to L2 meanwhile
    w.wait(k & nb1);
    const qs_real* hc = w.buf(k & nb1);                           // fields B_M .. B_LP at their own offsets
    qs_real* fac = q.sb + qs_blk(tile, N, k, NSB, lane);
    double* pcur = psm;                                          // P_{k+1}, p_{k+1} on entry; P_k, p_k on exit (in place)
    const double* pnx = psm;
    auto Pn = [&](int idx) { return QF(pnx, idx); };
    // gradient: g = ga + [B A]' (P_{k+1} rb + p_{k+1})
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
        y[i] = s + QF(pnx, 55 + i);
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
    // panel: columns 0..4 of the stage matrix, rows 0..14 (lower part)
    double pan[15][5];
#pragma unroll
    for (int i = 0; i < 15; ++i)
#pragma unroll
      for (int j = 0; j < 5; ++j)
        if (j <= i) pan[i][j] = QF(hc, H_M + tri(i, j)) + (k < N ? qs_y(i, j, dt, a2, Pn) : 0.0);
    // eliminate the control columns in place (LDL' form; a non-positive pivot zeroes the column, as BLASFEO dpotrf and
    // the oracle).  Rows are walked bottom-up so that the un-scaled column entries pan[c][j] of the rows above are
    // still available; afterwards pan[i][j] holds the multiplier t_ij (i > j) and pan[j][j] = 1/d_j.
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
    if (on) {
#pragma unroll
      for (int i = 0; i < 15; ++i)
#pragma unroll
        for (int j = 0; j < 5; ++j)
          if (j <= i) QF(fac, F_T + i * 5 + j) = pan[i][j];
#pragma unroll
      for (int i = 0; i < 15; ++i) QF(fac, F_LP + i) = g[i];
    }
#pragma unroll
    for (int i = 0; i < 10; ++i) QF(pcur, 55 + i) = g[5 + i];
    // P_k = trailing block - T_x D T_x', written in place over P_{k+1}: the vv block first, then vq, then qq -- an entry of
    // a later block only reads P_{k+1} entries of its own and of later blocks (qs_y), so nothing it needs is overwritten
    double sdx[10][5];
#pragma unroll
    for (int i = 5; i < 15; ++i)
#pragma unroll
      for (int j = 0; j < 5; ++j) sdx[i - 5][j] = pan[i][j] * dd[j];
    auto trail = [&](int i, int c) {
      double v = QF(hc, H_M + tri(i, c)) + (k < N ? qs_y(i, c, dt, a2, Pn) : 0.0);
#pragma unroll
      for (int j = 0; j < 5; ++j) v -= sdx[i - 5][j] * pan[c][j];
      QF(pcur, tri(i - 5, c - 5)) = v;
      if (on) QF(fac, F_P + tri(i - 5, c - 5)) = v;
    };
#pragma unroll
    for (int i = 10; i < 15; ++i)
#pragma unroll
      for (int c = 10; c <= i; ++c) trail(i, c);
#pragma unroll
    for (int i = 10; i < 15; ++i)
#pragma unroll
      for (int c = 5; c < 10; ++c) trail(i, c);
#pragma unroll
    for (int i = 5; i < 10; ++i)
#pragma unroll
      for (int c = 5; c <= i; ++c) trail(i, c);
    if (k == 0) {
      // factorise P_0 (kept per problem for the re-solves) and solve P_0 dx_0 = -p_0
      double m[10][10], gg[10];
#pragma unroll
      for (int i = 0; i < 10; ++i) {
        gg[i] = g[5 + i];
#pragma unroll
        for (int c = 0; c <= i; ++c) m[i][c] = QF(pcur, tri(i, c));
      }
#pragma unroll
      for (int j = 0; j < 10; ++j) {
        const double d = m[j][j];
        const double invd = d > 0.0 ? qs_rcp(d) : 0.0;
        m[j][j] = invd;
#pragma unroll
        for (int i = 9; i > j; --i) {       // bottom-up: the rows above still hold their un-scaled column entries
          const double t = m[i][j] * invd;
          gg[i] -= t * gg[j];
#pragma unroll
          for (int c = j + 1; c <= i; ++c) m[i][c] -= t * m[c][j];
          m[i][j] = t;
        }
      }
      if (on) {
#pragma unroll
        for (int i = 0; i < 10; ++i)
#pragma unroll
          for (int c = 0; c <= i; ++c) QF(pd, D_T0 + tri(i, c)) = m[i][c];
      }
#pragma unroll
      for (int i = 9; i >= 0; --i) {
        double acc = m[i][i] * gg[i];
#pragma unroll
        for (int c = i + 1; c < 10; ++c) acc += m[c][i] * dx[c];
        dx[i] = m[i][i] > 0.0 ? -acc : 0.0;
      }
    }
  }
  // forward substitution (affine direction): stages fetch RB, LP, T = fields [B_RB, B_WV)
  w.publish();
  w.sync();
  w.fetch_begin(0, B_WV - B_RB);
  w.fetch(0, 0, gsb, B_RB, B_WV - B_RB);
  for (int k = 0; k <= N; ++k) {
    w.sync();
    if (nb1 && k < N) { w.fetch_begin((k + 1) & 1, B_WV - B_RB); w.fetch((k + 1) & 1, 0, gsb + (size_t)(k + 1) * sstride, B_RB, B_WV - B_RB); }
    if (!nb1 && k > 0) { w.fetch_begin(0, B_WV - B_RB); w.fetch(0, 0, gsb + (size_t)k * sstride, B_RB, B_WV - B_RB); }
    if (!nb1 && k < N) w.prefetch(gsb + (size_t)(k + 1) * sstride, B_RB, B_WV - B_RB);
    w.wait(k & nb1);
    const qs_real* sb = w.buf(k & nb1) - (size_t)B_RB * TL;       // sb[f] valid for B_RB <= f < B_WV
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

// reduction of the step-length partials of one problem
SMPC_HD void qs_reduce_step(const QsBufs& q, int tile, int lane, double& alpha, double& s_lin, double& s_quad) {
  const int N = q.N;
  alpha = 1.0; s_lin = 0.0; s_quad = 0.0;
#pragma unroll 8
  for (int k = 0; k <= N; ++k) {
    const double* stp = q.stp + qs_blk(tile, N, k, NSTP, lane);
    alpha = fmin(alpha, QF(stp, S_ALPHA)); s_lin += QF(stp, S_LIN); s_quad += QF(stp, S_QUAD);
  }
}

// ric2: vector-only backward sweep, stage-0 solve and forward substitution with the multiplier steps, for the corrector
// right-hand side ga + v1 - sigma mu v2 AND, in the same pass, for the pure-centering right-hand side ga - sigma mu v2 that
// the conditional predictor-corrector falls back to (HPIPM: when the corrected step would more than double mu_aff).  Both
// share every factor load (T, P, WV, RB), the second vector rides in the latency shadow of the first, and the separate
// centering sweep of the earlier versions (a full sequential pass for the 1-80 % of the problems that asked for it)
// is gone; the arithmetic of each direction is unchanged.  The prologue turns the affine step statistics into sigma.
// Directions: corrector -> st (Z, PIM) and LP; centering -> st2 (Z, PIM) and LP2.
template <class W>
SMPC_HD void qs_ric2(const smpc_problem_t& P, const QsBufs& q, int tile, W& w) {
  const int N = q.N, lane = w.lane();
  const int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  const bool on = QF(pi, J_ACT) != 0;
  if (!w.any(on)) return;
  double* pd = q.pd + qs_pb(tile, NPD, lane);
  const double dt = P.dt, a2 = 0.5 * P.dt * P.dt;
  const qs_real* gsb = q.sb + qs_blk(tile, N, 0, NSB, 0);
  const size_t sstride = (size_t)NSB * TL;
  // backward stages fetch GA RB LP T WV = [B_GA, B_P) -> staging fields 0..124, and V1 V2 = [B_V1, NSB) -> 125..154
  const int n1 = B_P - B_GA, n2 = NSB - B_V1;
  const int nb1 = w.nbuf() - 1;
  w.fetch_begin(N & nb1, n1 + n2);
  w.fetch(N & nb1, 0, gsb + (size_t)N * sstride, B_GA, n1);
  w.fetch(N & nb1, n1, gsb + (size_t)N * sstride, B_V1, n2);
  double sigmu = 0.0;
  if (on) {
    double alpha, s_lin, s_quad;
    qs_reduce_step(q, tile, lane, alpha, s_lin, s_quad);
    const double mu = QF(pd, D_MU);
    const double mu_aff = mu + (alpha * s_lin + alpha * alpha * s_quad) / QF(pi, J_NC);
    double sigma = mu_aff / mu; sigma = sigma * sigma * sigma;
    sigmu = sigma * mu;
    QF(pd, D_MUAFF) = mu_aff; QF(pd, D_SIGMU) = sigmu;
  }
  double pn[2][10], dx[2][10];
#pragma unroll
  for (int v = 0; v < 2; ++v)
#pragma unroll
    for (int i = 0; i < 10; ++i) { pn[v][i] = 0.0; dx[v][i] = 0.0; }
  for (int k = N; k >= 0; --k) {
    w.sync();
    if (nb1 ? k > 0 : k < N) {
      const int kf = nb1 ? k - 1 : k;
      w.fetch_begin(kf & nb1, n1 + n2);
      w.fetch(kf & nb1, 0, gsb + (size_t)kf * sstride, B_GA, n1);
      w.fetch(kf & nb1, n1, gsb + (size_t)kf * sstride, B_V1, n2);
    }
    if (!nb1 && k > 0) { w.prefetch(gsb + (size_t)(k - 1) * sstride, B_GA, n1); w.prefetch(gsb + (size_t)(k - 1) * sstride, B_V1, n2); }
    w.wait(k & nb1);
    const qs_real* sb = w.buf(k & nb1) - (size_t)B_GA * TL;         // sb[f] valid for B_GA <= f < B_P
    const qs_real* vv = w.buf(k & nb1) - (size_t)(B_V1 - n1) * TL;  // vv[f] valid for B_V1 <= f < NSB
    qs_real* fac = q.sb + qs_blk(tile, N, k, NSB, lane);
    double g[2][15];
#pragma unroll
    for (int i = 0; i < 15; ++i) {
      const double ga = QF(sb, H_GA + i), s2 = sigmu * QF(vv, V_2 + i);
      g[0][i] = ga + QF(vv, V_1 + i) - s2;
      g[1][i] = ga + 0.0 - s2;
    }
    if (k < N) {
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        double y[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) y[i] = QF(sb, F_WV + i) + pn[v][i];
#pragma unroll
        for (int j = 0; j < 5; ++j) {
          g[v][j] += a2 * y[j] + dt * y[5 + j];
          g[v][5 + j] += y[j];
          g[v][10 + j] += dt * y[j] + y[5 + j];
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < 5; ++i) { g[0][i] = 0.0; g[1][i] = 0.0; }
    }
#pragma unroll
    for (int j = 0; j < 5; ++j)
#pragma unroll
      for (int i = j + 1; i < 15; ++i) { const double t = QF(sb, F_T + i * 5 + j); g[0][i] -= t * g[0][j]; g[1][i] -= t * g[1][j]; }
    if (on) {
#pragma unroll
      for (int i = 0; i < 15; ++i) { QF(fac, F_LP + i) = g[0][i]; QF(fac, F_LP2 + i) = g[1][i]; }
    }
#pragma unroll
    for (int v = 0; v < 2; ++v)
#pragma unroll
      for (int i = 0; i < 10; ++i) pn[v][i] = g[v][5 + i];
    if (k == 0) {
#pragma unroll
      for (int j = 0; j < 10; ++j)
#pragma unroll
        for (int i = j + 1; i < 10; ++i) { const double t = QF(pd, D_T0 + tri(i, j)); pn[0][i] -= t * pn[0][j]; pn[1][i] -= t * pn[1][j]; }
#pragma unroll
      for (int i = 9; i >= 0; --i) {
        const double invd = QF(pd, D_T0 + tri(i, i));
        double acc0 = invd * pn[0][i], acc1 = invd * pn[1][i];
#pragma unroll
        for (int c = i + 1; c < 10; ++c) { const double t = QF(pd, D_T0 + tri(c, i)); acc0 += t * dx[0][c]; acc1 += t * dx[1][c]; }
        dx[0][i] = invd > 0.0 ? -acc0 : 0.0;
        dx[1][i] = invd > 0.0 ? -acc1 : 0.0;
      }
    }
  }
  // forward: stages fetch RB LP T WV P LP2 = [B_RB, B_V1)
  w.publish();
  w.sync();
  w.fetch_begin(0, B_V1 - B_RB);
  w.fetch(0, 0, gsb, B_RB, B_V1 - B_RB);
  for (int k = 0; k <= N; ++k) {
    w.sync();
    if (nb1 && k < N) { w.fetch_begin((k + 1) & 1, B_V1 - B_RB); w.fetch((k + 1) & 1, 0, gsb + (size_t)(k + 1) * sstride, B_RB, B_V1 - B_RB); }
    if (!nb1 && k > 0) { w.fetch_begin(0, B_V1 - B_RB); w.fetch(0, 0, gsb + (size_t)k * sstride, B_RB, B_V1 - B_RB); }
    if (!nb1 && k < N) w.prefetch(gsb + (size_t)(k + 1) * sstride, B_RB, B_V1 - B_RB);
    w.wait(k & nb1);
    const qs_real* sb = w.buf(k & nb1) - (size_t)B_RB * TL;
    qs_real* st = q.st + qs_blk(tile, N, k, NIT, lane);
    qs_real* st2 = q.st2 + qs_blk(tile, N, k, NS2, lane);
    // multiplier step of the link k-1 -> k:  dpi = P_k dx_k + p_k
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      double s0 = 0.0, s1 = 0.0;
      if (k > 0) {
        s0 = QF(sb, F_LP + 5 + i); s1 = QF(sb, F_LP2 + 5 + i);
#pragma unroll
        for (int j = 0; j < 10; ++j) { const double pv = QF(sb, F_P + trs(i, j)); s0 += pv * dx[0][j]; s1 += pv * dx[1][j]; }
      }
      if (on) { QF(st, I_PIM + i) = s0; QF(st2, I_PIM + i) = s1; }
    }
    double du[2][5];
#pragma unroll
    for (int i = 0; i < 5; ++i) { du[0][i] = 0.0; du[1][i] = 0.0; }
    if (k < N) {
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const double tii = QF(sb, F_T + i * 5 + i);
        double ws0 = tii * QF(sb, F_LP + i), ws1 = tii * QF(sb, F_LP2 + i);
#pragma unroll
        for (int r = 0; r < 10; ++r) { const double t = QF(sb, F_T + (5 + r) * 5 + i); ws0 += t * dx[0][r]; ws1 += t * dx[1][r]; }
        du[0][i] = -ws0; du[1][i] = -ws1;
      }
#pragma unroll
      for (int c = 4; c >= 1; --c)
#pragma unroll
        for (int i = 0; i < c; ++i) { const double t = QF(sb, F_T + c * 5 + i); du[0][i] -= t * du[0][c]; du[1][i] -= t * du[1][c]; }
    }
    if (on) {
#pragma unroll
      for (int i = 0; i < 5; ++i) { QF(st, I_Z + i) = du[0][i]; QF(st2, I_Z + i) = du[1][i]; }
#pragma unroll
      for (int i = 0; i < 10; ++i) { QF(st, I_Z + 5 + i) = dx[0][i]; QF(st2, I_Z + 5 + i) = dx[1][i]; }
    }
    if (k < N) {
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        double nx[10];
#pragma unroll
        for (int j = 0; j < 5; ++j) {
          nx[j] = dx[v][j] + dt * dx[v][5 + j] + a2 * du[v][j] + QF(sb, H_RB + j);
          nx[5 + j] = dx[v][5 + j] + dt * du[v][j] + QF(sb, H_RB + 5 + j);
        }
#pragma unroll
        for (int j = 0; j < 10; ++j) dx[v][j] = nx[j];
      }
    }
  }
}

// ================================================================================================================
// step: recover (dlam, dt, dslack) of every row from dz, step-length partials.   thread = (problem, stage)
//   mode 0 (affine): stores dlam*dt per slot and the corrector gradient terms v1, v2
//   mode 1 / 2 (corrector / centering): stores the step
//
// Operand source.  qs_step reads its stage block (iterate, step or centering direction, products, record) through a policy S:
//   S.it(c, f), S.st(c, f), S.st2(c, f), S.prod(c, f), S.rec(c, f)   field f of that block, widened to fp64
//   S.acquire(c) / S.release(c)                                       chunk c is about to be read / has been read for the last time
// The chunks c = 0 .. QSC_N - 1 follow the load phases in the order they run (table qs_sp below).  QsStepGlobal reads global memory
// (acquire / release are no-ops); the staged kernels of qp.cu read a per-warp ring of chunks that bulk copies fill ahead of the
// arithmetic.  Every lane runs the same instructions on the same values in both: a problem's result does not depend on the source.
// Stores go to global memory in both.
// ================================================================================================================
enum { QA_NONE = 0, QA_IT, QA_ST, QA_ST2, QA_REC, QA_PROD };
struct QsPiece { int a, f0, n; };   // fields [f0, f0 + n) of one array of the stage block
enum { QSC_N = 16, QSC_PIECES = 7 };
// both sides of the row slots [s0, s0 + n): lam (lower, upper), t (lower, upper), and in mode 1 the products
SMPC_HD constexpr QsPiece qs_sp_rows(int mode, int s0, int n, int i) {
  return i < 4 ? QsPiece{QA_IT, ((i & 2) ? I_T : I_LAM) + (i & 1) * QNR + s0, n}
               : (mode == 1 && i < 6) ? QsPiece{QA_PROD, (i & 1) * QNR + s0, n} : QsPiece{QA_NONE, 0, 0};
}
// piece i of chunk c in `mode` (n = 0: past the last piece).  The record ranges are cut so that no chunk exceeds 36 fields: the torque
// rows in pieces of two rows, each with the five torque values the rows are compared against; the Jacobians are fetched again for the
// corrector terms of mode 0 (they were read three phases earlier, from L2 by then).
SMPC_HD constexpr QsPiece qs_sp(int mode, int c, int i) {
  constexpr QsPiece no{QA_NONE, 0, 0};
  switch (c) {
    case 0: return i == 0 ? QsPiece{QA_IT, I_Z, 15} : i == 1 ? QsPiece{mode == 2 ? QA_ST2 : QA_ST, I_Z, 15} : no;   // z, dz
    case 1: return i == 0 ? QsPiece{QA_REC, SMPC_REC_X, 5} : qs_sp_rows(mode, 0, 5, i - 1);                     // box rows 0-4
    case 2: return i == 0 ? QsPiece{QA_REC, SMPC_REC_X + 5, 5} : qs_sp_rows(mode, 5, 5, i - 1);                 // box rows 5-9
    case 3: return i == 0 ? QsPiece{QA_REC, SMPC_REC_TAU, 35} : no;                                             // tau, rows 0-1 of d tau
    case 4: return i == 0 ? QsPiece{QA_REC, SMPC_REC_TAU, 5} : i == 1 ? QsPiece{QA_REC, SMPC_REC_JTAU + 30, 30} : no;
    case 5: return i == 0 ? QsPiece{QA_REC, SMPC_REC_TAU, 5} : i == 1 ? QsPiece{QA_REC, SMPC_REC_JTAU + 60, 15} : no;
    case 6: return i == 0 ? QsPiece{QA_REC, SMPC_REC_DIST, 36} : no;                                            // capsule rows
    case 7: return i == 0 ? QsPiece{QA_REC, SMPC_REC_NN, 11} : no;                                              // viability row
    case 8: return qs_sp_rows(mode, 10, 5, i);                                                                  // torque slots
    case 9: return mode == 0 && i == 0 ? QsPiece{QA_REC, SMPC_REC_JTAU, 30} : no;
    case 10: return mode == 0 && i == 0 ? QsPiece{QA_REC, SMPC_REC_JTAU + 30, 30} : no;
    case 11: return mode == 0 && i == 0 ? QsPiece{QA_REC, SMPC_REC_JTAU + 60, 15} : no;
    case 12: return qs_sp_rows(mode, 15, 6, i);                                                                 // capsule slots
    case 13: return mode == 0 && i == 0 ? QsPiece{QA_REC, SMPC_REC_JDIST, 30} : no;
    case 14:                                                                                                    // viability slots, slacks
      return i == 0 ? QsPiece{QA_REC, SMPC_REC_NN, 11} : i == 1 ? QsPiece{QA_IT, I_LAM + 21, 1} : i == 2 ? QsPiece{QA_IT, I_LAM + QNR + 21, 1}
           : i == 3 ? QsPiece{QA_IT, I_T + 21, 1} : i == 4 ? QsPiece{QA_IT, I_T + QNR + 21, 8}   // t (upper) + the six slack fields
           : mode == 1 && i == 5 ? QsPiece{QA_PROD, 21, 1} : mode == 1 && i == 6 ? QsPiece{QA_PROD, QNR + 21, 3} : no;
    case 15: return mode == 2 && i == 0 ? QsPiece{QA_ST2, I_PIM, 10} : no;                                     // dpi of the centering direction
    default: return no;
  }
}
static_assert(I_T + QNR + 21 + 8 <= NIT && I_SLK + 6 <= I_T + QNR + 21 + 8, "viability chunk covers the slacks");
SMPC_HD constexpr int qs_sp_esz(int a) { return a == QA_IT ? (int)sizeof(double) : (int)sizeof(qs_real); }
SMPC_HD constexpr int qs_sp_bytes(const QsPiece& p) { return p.n * TL * qs_sp_esz(p.a); }
SMPC_HD constexpr int qs_chunk_bytes(int mode, int c) {
  int b = 0;
  for (int i = 0; i < QSC_PIECES; ++i) b += qs_sp_bytes(qs_sp(mode, c, i));
  return b;
}
SMPC_HD constexpr int qs_chunk_max_bytes() {
  int m = 0;
  for (int mode = 0; mode < 3; ++mode)
    for (int c = 0; c < QSC_N; ++c) m = qs_chunk_bytes(mode, c) > m ? qs_chunk_bytes(mode, c) : m;
  return m;
}
// byte offset of field f of array a inside chunk c (layout [field][lane], pieces in table order); -1: not in the chunk
SMPC_HD constexpr int qs_chunk_off(int mode, int c, int a, int f) {
  int off = 0;
  for (int i = 0; i < QSC_PIECES; ++i) {
    const QsPiece p = qs_sp(mode, c, i);
    if (p.a == a && f >= p.f0 && f < p.f0 + p.n) return off + (f - p.f0) * TL * qs_sp_esz(a);
    off += qs_sp_bytes(p);
  }
  return -1;
}
// chunks the stage does not use (its rows are absent) are skipped: nothing is fetched
SMPC_HD bool qs_chunk_on(int c, const StageFlags& F) {
  return (c >= 3 && c <= 5) || (c >= 8 && c <= 11) ? F.tau : (c == 6 || c == 12 || c == 13) ? F.dist : (c == 7 || c == 14) ? F.nn : true;
}

struct QsStepGlobal {
  const qs_real* rec_;
  const double* it_;
  const qs_real* st_;
  const qs_real* st2_;
  const qs_real* prod_;
  SMPC_HD QsStepGlobal(const QsBufs& q, int tile, int lane, int k, int kk)
      : rec_(q.rec + qs_blk(tile, q.N, k, REC, lane)), it_(q.it[kk & 1] + qs_blk(tile, q.N, k, NIT, lane)), st_(q.st + qs_blk(tile, q.N, k, NIT, lane)),
        st2_(q.st2 + qs_blk(tile, q.N, k, NS2, lane)), prod_(q.prod + qs_blk(tile, q.N, k, NPROD, lane)) {}
  SMPC_HD void acquire(int) const {}
  SMPC_HD void release(int) const {}
  SMPC_HD double it(int, int f) const { return QF(it_, f); }
  SMPC_HD double st(int, int f) const { return QF(st_, f); }
  SMPC_HD double st2(int, int f) const { return QF(st2_, f); }
  SMPC_HD double prod(int, int f) const { return QF(prod_, f); }
  SMPC_HD double rec(int, int f) const { return QF(rec_, f); }
};

template <class S>
SMPC_HD void qs_step(const smpc_problem_t& P, const QsBufs& q, int tile, int lane, int k, int kk, int mode, S& src) {
  const int N = q.N;
  const int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  if (!QF(pi, J_ACT)) return;
  if (mode == 2 && !QF(pi, J_REDO)) return;
  const double* pd = q.pd + qs_pb(tile, NPD, lane);
  const int rrec = QF(pi, J_R);
  const double sigmu = mode == 0 ? 0.0 : QF(pd, D_SIGMU);
  qs_real* st = q.st + qs_blk(tile, N, k, NIT, lane);
  qs_real* prod = q.prod + qs_blk(tile, N, k, NPROD, lane);
  const StageFlags F = qs_flags(P, k);
  double z[15], dz[15];
  src.acquire(0);
  if (mode == 2) {
    // the centering direction was computed by ric2 next to the corrector: it becomes the step of this problem
#pragma unroll
    for (int i = 0; i < 15; ++i) { z[i] = src.it(0, I_Z + i); dz[i] = src.st2(0, I_Z + i); }
  } else {
#pragma unroll
    for (int i = 0; i < 15; ++i) { z[i] = src.it(0, I_Z + i); dz[i] = src.st(0, I_Z + i); }
  }
  src.release(0);
  // step length = min over the slots of lam / (-dlam), t / (-dt) (negative steps only), kept as a fraction an / ad and
  // compared by cross-multiplication: one division per thread instead of two per slot
  double an = 1.0, ad = 1.0, s_lin = 0.0, s_quad = 0.0;
  auto ratio = [&](double num, double neg_den) { if (neg_den < 0.0 && num * ad < an * (-neg_den)) { an = num; ad = -neg_den; } };
  double v1[15], v2[15];
#pragma unroll
  for (int i = 0; i < 15; ++i) { v1[i] = 0.0; v2[i] = 0.0; }

  // Loads and stores are kept in separate phases per row group (see qs_prep).
  // one side of a hard row.  e1 / e2: this side's contribution to the corrector terms (signed)
  auto side = [&](int slot, double sgn, double az, double adz, double bnd, double lam, double t, double pr, double& e1, double& e2) {
    const double r = t - sgn * (az - bnd);
    const double rm = qs_rm(mode, lam * t, pr, sigmu);
    const double it_ = 1.0 / t;
    const double dtt = sgn * adz - r;
    const double dl = -(rm + lam * dtt) * it_;
    ratio(lam, dl); ratio(t, dtt);
    s_lin += lam * dtt + t * dl; s_quad += dl * dtt;
    if (mode == 0) { const double pp = dl * dtt; QF(prod, slot) = pp; e1 += sgn * pp * it_; e2 += sgn * it_; }
    else { QF(st, I_LAM + slot) = dl; QF(st, I_T + slot) = dtt; }
  };
  // box rows
  {
    double lo[10], hi[10], bl[20], bt[20], bp[20];
#pragma unroll
    for (int j = 0; j < 10; ++j) {
      const int c = j < 5 ? 1 : 2;
      if (j == 0) src.acquire(1);
      if (j == 5) { src.release(1); src.acquire(2); }
      qs_box_x(P, q, tile, lane, k, j, src.rec(c, SMPC_REC_X + j), QF(pd, D_X0 + j), rrec, lo[j], hi[j]);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        bl[h * 10 + j] = src.it(c, I_LAM + h * QNR + j); bt[h * 10 + j] = src.it(c, I_T + h * QNR + j);
        bp[h * 10 + j] = mode == 1 ? src.prod(c, h * QNR + j) : 0.0;
      }
    }
    src.release(2);
#pragma unroll
    for (int j = 0; j < 10; ++j) {
      double e1 = 0.0, e2 = 0.0;
      side(j, 1.0, z[5 + j], dz[5 + j], lo[j], bl[j], bt[j], bp[j], e1, e2);
      side(QNR + j, -1.0, z[5 + j], dz[5 + j], hi[j], bl[10 + j], bt[10 + j], bp[10 + j], e1, e2);
      v1[5 + j] += e1; v2[5 + j] += e2;
    }
  }
  // general rows: row products of z and dz, bounds (loads only)
  double azg[12], adg[12], glo[12], ghi[12];
#pragma unroll
  for (int r = 0; r < 12; ++r) { azg[r] = adg[r] = glo[r] = ghi[r] = 0.0; }
  if (F.tau) {
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      const int cj = 3 + r / 2;        // chunk of d tau row r (with tau)
      if (r == 0) src.acquire(3);
      if (r == 2 || r == 4) { src.release(cj - 1); src.acquire(cj); }
      double az = 0.0, adz = 0.0;
#pragma unroll
      for (int c = 0; c < 15; ++c) { const double jv = src.rec(cj, SMPC_REC_JTAU + r * 15 + c); az += jv * z[c]; adz += jv * dz[c]; }
      const double v = src.rec(cj, SMPC_REC_TAU + r);
      azg[r] = az; adg[r] = adz; glo[r] = P.tau_min[r] - v; ghi[r] = P.tau_max[r] - v;
    }
    src.release(5);
  } else {
    for (int c = 3; c <= 5; ++c) { src.acquire(c); src.release(c); }
  }
  src.acquire(6);
  if (F.dist) {
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      double az = 0.0, adz = 0.0;
#pragma unroll
      for (int c = 0; c < 5; ++c) { const double jv = src.rec(6, SMPC_REC_JDIST + p * 5 + c); az += jv * z[5 + c]; adz += jv * dz[5 + c]; }
      const double v = src.rec(6, SMPC_REC_DIST + p);
      azg[5 + p] = az; adg[5 + p] = adz; glo[5 + p] = P.pair_lo_ocp[p] - v; ghi[5 + p] = P.pair_hi - v;
    }
  }
  src.release(6);
  src.acquire(7);
  if (F.nn) {
    double az = 0.0, adz = 0.0;
#pragma unroll
    for (int c = 0; c < 10; ++c) { const double jv = src.rec(7, SMPC_REC_JNN + c); az += jv * z[5 + c]; adz += jv * dz[5 + c]; }
    const double v = src.rec(7, SMPC_REC_NN);
    azg[11] = az; adg[11] = adz; glo[11] = 0.0 - v; ghi[11] = 1e6 - v;
  }
  src.release(7);
  if (F.tau) {
    double gl[10], gt[10], gp[10];
    src.acquire(8);
#pragma unroll
    for (int r = 0; r < 5; ++r)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int slot = h * QNR + 10 + r;
        gl[h * 5 + r] = src.it(8, I_LAM + slot); gt[h * 5 + r] = src.it(8, I_T + slot); gp[h * 5 + r] = mode == 1 ? src.prod(8, slot) : 0.0;
      }
    src.release(8);
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      const int cj = 9 + r / 2;        // chunk of d tau row r (corrector terms, mode 0)
      if (r == 0) src.acquire(9);
      if (r == 2 || r == 4) { src.release(cj - 1); src.acquire(cj); }
      double e1 = 0.0, e2 = 0.0;
      side(10 + r, 1.0, azg[r], adg[r], glo[r], gl[r], gt[r], gp[r], e1, e2);
      side(QNR + 10 + r, -1.0, azg[r], adg[r], ghi[r], gl[5 + r], gt[5 + r], gp[5 + r], e1, e2);
      if (mode == 0) {
#pragma unroll
        for (int c = 0; c < 15; ++c) { const double jv = src.rec(cj, SMPC_REC_JTAU + r * 15 + c); v1[c] += jv * e1; v2[c] += jv * e2; }
      }
    }
    src.release(11);
  } else {
    for (int c = 8; c <= 11; ++c) { src.acquire(c); src.release(c); }
  }
  src.acquire(12);
  if (F.dist) {
    double gl[12], gt[12], gp[12];
#pragma unroll
    for (int p = 0; p < 6; ++p)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int slot = h * QNR + 15 + p;
        gl[h * 6 + p] = src.it(12, I_LAM + slot); gt[h * 6 + p] = src.it(12, I_T + slot); gp[h * 6 + p] = mode == 1 ? src.prod(12, slot) : 0.0;
      }
    src.release(12);
    src.acquire(13);
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      double e1 = 0.0, e2 = 0.0;
      side(15 + p, 1.0, azg[5 + p], adg[5 + p], glo[5 + p], gl[p], gt[p], gp[p], e1, e2);
      side(QNR + 15 + p, -1.0, azg[5 + p], adg[5 + p], ghi[5 + p], gl[6 + p], gt[6 + p], gp[6 + p], e1, e2);
      if (mode == 0) {
#pragma unroll
        for (int c = 0; c < 5; ++c) { const double jv = src.rec(13, SMPC_REC_JDIST + p * 5 + c); v1[5 + c] += jv * e1; v2[5 + c] += jv * e2; }
      }
    }
  } else {
    src.release(12);
    src.acquire(13);
  }
  src.release(13);
  src.acquire(14);
  if (F.nn) {
    const double az = azg[11], adz = adg[11];
    const double v = src.rec(14, SMPC_REC_NN);
    double e1 = 0.0, e2 = 0.0;
    if (!F.soft) {
      const double l0 = src.it(14, I_LAM + 21), t0 = src.it(14, I_T + 21), p0 = mode == 1 ? src.prod(14, 21) : 0.0;
      const double l1 = src.it(14, I_LAM + QNR + 21), t1 = src.it(14, I_T + QNR + 21), p1 = mode == 1 ? src.prod(14, QNR + 21) : 0.0;
      side(21, 1.0, az, adz, 0.0 - v, l0, t0, p0, e1, e2);
      side(QNR + 21, -1.0, az, adz, 1e6 - v, l1, t1, p1, e1, e2);
      if (mode != 0) {
#pragma unroll
        for (int h = 0; h < 6; ++h) QF(st, I_SLK + h) = 0.0;
      }
    } else {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int slot = h * QNR + 21;
        const double sgn = h ? -1.0 : 1.0, bnd = h ? 1e6 - v : 0.0 - v;
        const double lam = src.it(14, I_LAM + slot), t = src.it(14, I_T + slot);
        const double sl = src.it(14, I_SLK + h), ls = src.it(14, I_SLK + 2 + h), ts = src.it(14, I_SLK + 4 + h);
        const double r = t - (sgn * (az - bnd) + sl);
        const double pr = mode == 1 ? src.prod(14, slot) : 0.0, spr = mode == 1 ? src.prod(14, 44 + h) : 0.0;
        const double rm = qs_rm(mode, lam * t, pr, sigmu);
        const double it_ = 1.0 / t;
        const double G = lam * it_;
        const double c = (rm - lam * r) * it_;
        const double rsl = ts - sl;
        const double rgs = F.zpen - lam - ls;
        const double rms = qs_rm(mode, ls * ts, spr, sigmu);
        const double its = 1.0 / ts;
        const double Gs = ls * its;
        const double cs = (rms - ls * rsl) * its;
        const double W = 1.0 / (G + Gs);
        const double ds = -(rgs + c + cs + sgn * G * adz) * W;
        const double dts = ds - rsl;
        const double dls = -(rms + ls * dts) * its;
        ratio(ls, dls); ratio(ts, dts);
        s_lin += ls * dts + ts * dls; s_quad += dls * dts;
        const double dtt = sgn * adz + ds - r;
        const double dl = -(rm + lam * dtt) * it_;
        ratio(lam, dl); ratio(t, dtt);
        s_lin += lam * dtt + t * dl; s_quad += dl * dtt;
        if (mode == 0) {
          const double pp = dl * dtt, sp = dls * dts;
          QF(prod, slot) = pp; QF(prod, 44 + h) = sp;
          // d cc = (1 - G W) d c - G W d cs  with  d c = (pp - sigmu)/t,  d cs = (sp - sigmu)/ts
          const double gw = G * W;
          e1 += sgn * ((1.0 - gw) * pp * it_ - gw * sp * its);
          e2 += sgn * ((1.0 - gw) * it_ - gw * its);
        } else {
          QF(st, I_LAM + slot) = dl; QF(st, I_T + slot) = dtt;
          QF(st, I_SLK + h) = ds; QF(st, I_SLK + 2 + h) = dls; QF(st, I_SLK + 4 + h) = dts;
        }
      }
    }
    if (mode == 0) {
#pragma unroll
      for (int c = 0; c < 10; ++c) { const double jv = src.rec(14, SMPC_REC_JNN + c); v1[5 + c] += jv * e1; v2[5 + c] += jv * e2; }
    }
  }
  src.release(14);
  if (mode == 0) {
    qs_real* vv = q.sb + qs_blk(tile, N, k, NV, lane);
    if (k == N) {
#pragma unroll
      for (int i = 0; i < 5; ++i) { v1[i] = 0.0; v2[i] = 0.0; }
    }
#pragma unroll
    for (int i = 0; i < 15; ++i) { QF(vv, V_1 + i) = v1[i]; QF(vv, V_2 + i) = v2[i]; }
  }
  if (mode == 2) {
    // (dz, dpi) of the step block <- centering direction (after every load of this thread, see the note on load / store phases)
    double dpi[10];
    src.acquire(15);
#pragma unroll
    for (int j = 0; j < 10; ++j) dpi[j] = src.st2(15, I_PIM + j);
    src.release(15);
#pragma unroll
    for (int i = 0; i < 15; ++i) QF(st, I_Z + i) = dz[i];
#pragma unroll
    for (int j = 0; j < 10; ++j) QF(st, I_PIM + j) = dpi[j];
  }
  double* stp = q.stp + qs_blk(tile, N, k, NSTP, lane);
  QF(stp, S_ALPHA) = an / ad; QF(stp, S_LIN) = s_lin; QF(stp, S_QUAD) = s_quad;
}
SMPC_HD void qs_step(const smpc_problem_t& P, const QsBufs& q, int tile, int lane, int k, int kk, int mode) {
  QsStepGlobal src(q, tile, lane, k, kk);
  qs_step(P, q, tile, lane, k, kk, mode, src);
}

// ================================================================================================================
// red: step length of the corrector; conditional predictor-corrector (fall back to pure centering when the corrected
// step would more than double mu_aff).   thread = problem.   after_redo: second call, for the problems that re-solved.
// ================================================================================================================
SMPC_HD void qs_red(const smpc_problem_t& P, const QsBufs& q, int tile, int lane, bool after_redo) {
  int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  if (!QF(pi, J_ACT)) return;
  if (after_redo && !QF(pi, J_REDO)) return;
  double* pd = q.pd + qs_pb(tile, NPD, lane);
  double alpha, s_lin, s_quad;
  qs_reduce_step(q, tile, lane, alpha, s_lin, s_quad);
  int redo = 0;
  if (!after_redo && P.qp_cond_pred_corr) {
    const double mu_corr = QF(pd, D_MU) + (alpha * s_lin + alpha * alpha * s_quad) / QF(pi, J_NC);
    if (mu_corr > 2.0 * QF(pd, D_MUAFF)) redo = 1;
  }
  QF(pi, J_REDO) = redo;
  QF(pd, D_ALPHA) = alpha;
  QF(pd, D_STEP) = 0.995 * alpha;
}

// per-problem initialisation of one solve.   thread = problem (lane of a tile; b = 32 tile + lane may be >= B: padding)
SMPC_HD void qs_init(const QsBufs& q, int tile, int lane, int B, const double* x0, const int32_t* r, const uint8_t* act) {
  const int b = (q.tile0 + tile) * TL + lane;
  int32_t* pi = q.pi + qs_pb(tile, NPI, lane);
  double* pd = q.pd + qs_pb(tile, NPD, lane);
  const bool on = b < B && (!act || act[b]);
  QF(pi, J_ACT) = on ? 1 : 0; QF(pi, J_ITER) = 0; QF(pi, J_QST) = 0; QF(pi, J_REDO) = 0; QF(pi, J_NC) = 1; QF(pi, J_ITBUF) = 0;
  QF(pi, J_R) = b < B ? r[b] : 0; QF(pi, J_B) = b < B ? b : -1; QF(pi, J_FIN) = 0;
  for (int j = 0; j < NX; ++j) QF(pd, D_X0 + j) = b < B ? x0[(size_t)b * NX + j] : 0.0;
  QF(pd, D_MU) = 0.0; QF(pd, D_MUAFF) = 0.0; QF(pd, D_SIGMU) = 0.0; QF(pd, D_ALPHA) = 1.0; QF(pd, D_STEP) = 0.0;
}

// Host-side sequencing of one batched solve of one group of tiles; BK launches the phases (CUDA kernels in qp.cu, plain
// loops in tests/emu).  One IPM iteration = ctl, ric1, step<0>, ric2, step<1>, red, [step<2>, red], [compaction], prep of the
// next iterate.  The host needs two numbers per iteration -- problems still active, problems that asked for the centering
// re-solve -- to stop, to pick between kernel forms that give identical results, and to decide on a compaction.
//   depth = 0   the host waits for the counters of every iteration before it queues the next one (one round trip per iteration;
//               step<2> / red only when some problem asked for them)
//   depth > 0   the host runs up to `depth` iterations ahead of the counters it has seen: it polls, blocks only when `depth`
//               iterations are in flight, and queues step<2> / red unconditionally (they filter per problem); every kernel of an
//               iteration queued past the end of the solve finds no active problem and exits.  The GPU never waits for the host.
// Several groups are driven round-robin so that the latency-bound Riccati sweeps of one group overlap the bandwidth-bound
// stage-parallel kernels of the others.
template <class BK>
struct QsLoop {
  BK& bk;
  int kk = 0;
  int depth = 0;
  int kk_seen = -1;              // newest iteration whose counters the host has read
  bool done = false;
  explicit QsLoop(BK& b, int depth_ = 0) : bk(b), depth(depth_) {}
  void issue() {
    bk.ctl(kk);
    bk.ric1();
    bk.step(kk, 0);
    bk.ric2();
    bk.step(kk, 1);
    bk.red(false);
    if (depth > 0) { bk.step(kk, 2); bk.red(true); }
    bk.request_counters(kk);
  }
  void start() {
    bk.init(); bk.prep(0);
    if (bk.solo(0)) { bk.final(); done = true; return; }      // small batch: the backend runs the whole solve on its own
    issue();
  }
  void advance() {
    int n_active = 0, n_redo = 0;
    if (depth == 0) {
      bk.wait_counters(kk, true, n_active, n_redo);
      kk_seen = kk;
      if (n_active == 0) { bk.final(); done = true; return; }
      if (n_redo > 0) { bk.step(kk, 2); bk.red(true); }
    } else {
      while (kk_seen < kk) {
        if (!bk.wait_counters(kk_seen + 1, kk - kk_seen >= depth, n_active, n_redo)) break;
        ++kk_seen;
        if (n_active == 0) { bk.final(); done = true; return; }
      }
    }
    bk.compact(kk);              // (the backend decides; a no-op for most iterations)
    ++kk;
    bk.prep(kk);
    if (bk.solo(kk)) { bk.final(); done = true; return; }     // few problems left: the backend finishes the solve on its own (qp.cu: solo kernel)
    issue();
  }
};

template <class BK>
int qs_drive(BK* groups, int n_groups, int depth = 0) {
  QsLoop<BK>* loops[8];
  for (int g = 0; g < n_groups; ++g) { loops[g] = new QsLoop<BK>(groups[g], depth); loops[g]->start(); }
  int kmax = 0;
  for (bool any = true; any;) {
    any = false;
    for (int g = 0; g < n_groups; ++g)
      if (!loops[g]->done) { loops[g]->advance(); any = any || !loops[g]->done; }
  }
  for (int g = 0; g < n_groups; ++g) { kmax = loops[g]->kk > kmax ? loops[g]->kk : kmax; delete loops[g]; }
  return kmax;
}

// Device-side sequencing of one solve (a solve captured into a CUDA graph: the host cannot read counters, DESIGN §3.2).  The
// iteration index lives in device memory (*kk); one iteration is the run-ahead order of QsLoop::issue with step<2> / red queued
// unconditionally, followed by the loop step below and the prep of the next iterate.  The backend repeats the body while the loop
// step says so: qp.cu as a conditional WHILE node of the graph, tests/graph_loop_host.cpp as a plain loop.
// Loop step (one thread): reads the active count of iteration *kk, advances *kk, and returns whether the body runs again.
SMPC_HD bool qs_loop_continue(int n_active, int kk, int iter_max) { return n_active > 0 && kk < iter_max; }
SMPC_HD bool qs_loop_step(const int* counters, int* kk, int iter_max) {
  const int k = *kk;
  *kk = k + 1;
  return qs_loop_continue(counters[2 * k], k, iter_max);
}

template <class BK>
void qs_graph_body(BK& bk) {
  bk.ctl(0);
  bk.ric1();
  bk.step(0, 0);
  bk.ric2();
  bk.step(0, 1);
  bk.red(false);
  bk.step(0, 2);
  bk.red(true);
  bk.loop_step();
  bk.prep(0);          // the iterate of the new *kk
}

// init and prep(0) as in QsLoop::start; the solo kernel when the backend takes it (decided from what the host knows at iteration 0),
// else the device-side loop; then final
template <class BK>
void qs_graph_drive(BK& bk) {
  bk.init(); bk.prep(0);
  if (!bk.solo(0)) bk.loop(qs_graph_body<BK>);
  bk.final();
}

}  // inline namespace QS_FLAVOUR
}  // namespace smpc
