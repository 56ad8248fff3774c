// TEST HARNESS -- host build of the two schedules of one batched QP solve (safe_mpc_b200/csrc/qp_split.cuh): the host-driven loop qs_drive
// (the eager path, depth 0: the host reads the counters of every iteration) and qs_graph_drive, the schedule of a solve captured into a CUDA
// graph: no compaction, fixed kernel forms, step<2> / red(true) in every iteration, the iteration index in "device" memory and the loop
// repeated while the shared loop step qs_loop_step says so.  Every phase runs as plain loops over (tile, stage, lane).  Not part of the product.
#include <cstring>
#include <vector>

#include "../safe_mpc_b200/csrc/qp_split.cuh"

using namespace smpc;

namespace {
// host stand-in of the staged copies of the Riccati sweeps (copies complete at once)
struct HostStage {
  int ln, nfb, nb = 2;
  std::vector<qs_real> mem;
  HostStage(int lane_, int nfb_) : ln(lane_), nfb(nfb_), mem((size_t)2 * nfb_ * TL, (qs_real)0) {}
  int nbuf() const { return nb; }
  int lane() const { return ln; }
  bool any(bool v) const { return v; }
  void sync() const {}
  qs_real* buf(int b) { return mem.data() + (size_t)b * nfb * TL + ln; }
  void fetch_begin(int, int) {}
  void fetch(int b, int dst_field, const qs_real* gblock, int src_field, int nfields) {
    std::memcpy(mem.data() + ((size_t)b * nfb + dst_field) * TL, gblock + (size_t)src_field * TL, (size_t)nfields * TL * sizeof(qs_real));
  }
  void wait(int) {}
  void publish() const {}
  void prefetch(const qs_real*, int, int) const {}
};

struct Backend {
  const smpc_problem_t& P;
  QsBufs q;
  int B, T, N;
  const double* x0; const int32_t* r; const uint8_t* act;
  double *xt, *ut; int32_t *status, *qp_iter, *qp_status; double* qp_res;
  std::vector<double> psm = std::vector<double>(65 * TL, 0.0);
  std::vector<int> counters;        // [2 (iter_max + 2)]: active / redo per iteration, as the kernels count them
  int kk_dev = 0;                   // the device-resident iteration of the captured schedule
  bool in_body = false;             // inside the loop body: every phase takes its iteration from kk_dev
  bool cond = false;
  int n_body = 0;                   // loop bodies run
  int kk_last = 0;
  int it(int kk) const { return in_body ? kk_dev : kk; }
  template <class F> void each_stage(F f) { for (int t = 0; t < T; ++t) for (int k = 0; k <= N; ++k) for (int l = 0; l < TL; ++l) f(t, l, k); }
  template <class F> void each_problem(F f) { for (int t = 0; t < T; ++t) for (int l = 0; l < TL; ++l) f(t, l); }
  void init() {
    counters.assign((size_t)2 * (P.qp_iter_max + 2), 0);
    each_problem([&](int t, int l) { qs_init(q, t, l, B, x0, r, act); });
  }
  void prep(int kk) {
    const int k0 = it(kk);
    std::vector<double> jsm((size_t)PREP_SCRATCH * TL, 0.0);
    each_stage([&](int t, int l, int k) {
      if (k0 == 0 && !in_body) qs_prep<true>(P, q, t, l, k, k0, jsm.data() + l); else qs_prep<false>(P, q, t, l, k, k0, jsm.data() + l);
    });
  }
  void ctl(int kk) {
    const int k0 = it(kk);
    kk_last = k0;
    each_problem([&](int t, int l) { if (qs_ctl(P, q, t, l, k0, status, qp_iter, qp_status, qp_res)) ++counters[2 * k0]; });
  }
  void ric1() { each_problem([&](int t, int l) { HostStage w(l, RIC1_STAGE_FIELDS); qs_ric1(P, q, t, w, psm.data() + l); }); }
  void ric2() { each_problem([&](int t, int l) { HostStage w(l, RIC2_STAGE_FIELDS); qs_ric2(P, q, t, w); }); }
  void step(int kk, int mode) { const int k0 = it(kk); each_stage([&](int t, int l, int k) { qs_step(P, q, t, l, k, k0, mode); }); }
  void red(bool after) {
    each_problem([&](int t, int l) {
      qs_red(P, q, t, l, after);
      const int32_t* pi = q.pi + qs_pb(t, NPI, l);
      if (!after && QF(pi, J_ACT) && QF(pi, J_REDO)) ++counters[2 * kk_last + 1];
    });
  }
  void final() { each_stage([&](int t, int l, int k) { const int b = qs_final(q, t, l, k, act, B, status, xt, ut); if (b >= 0) status[b] = 1; }); }
  bool solo(int) { return false; }
  void compact(int) {}
  void request_counters(int) {}
  bool wait_counters(int kk, bool, int& na, int& nr) { na = counters[2 * kk]; nr = counters[2 * kk + 1]; return true; }
  // the conditional WHILE node: the reset kernel, then the body while the condition holds
  template <class F> void loop(F body) {
    kk_dev = 0; cond = true;
    while (cond) { in_body = true; body(*this); in_body = false; ++n_body; }
  }
  void loop_step() { cond = qs_loop_step(counters.data(), &kk_dev, P.qp_iter_max); }
};
}  // namespace

// One batched solve in either schedule.  rec: [B][N+1][REC] (caller layout), x0: [B][10], r: [B], act: [B] or NULL.  graph = 0: qs_drive at
// depth 0, 1: qs_graph_drive.  Returns the number of loop bodies run (graph) or the iterations of the host loop.
extern "C" int graph_loop_solve(const smpc_problem_t* P, int B, const double* rec, const double* x0, const int32_t* r, const uint8_t* act, int graph,
                                double* xt, double* ut, int32_t* status, int32_t* qp_iter, int32_t* qp_status, double* qp_res) {
  const int N = P->N, T = (B + TL - 1) / TL;
  const size_t S = (size_t)T * (N + 1) * TL;
  std::vector<qs_real> vrec(S * REC, (qs_real)0), st(S * NIT, (qs_real)0), st2(S * NS2, (qs_real)0), prod(S * NPROD, (qs_real)0), sb(S * NSB, (qs_real)0);
  std::vector<double> it0(S * NIT, 0.0), it1(S * NIT, 0.0), res(S * NRES, 0.0), stp(S * NSTP, 0.0), pd((size_t)T * NPD * TL, 0.0);
  std::vector<int32_t> pi32((size_t)T * NPI * TL, 0);
  for (int b = 0; b < B; ++b)
    for (int k = 0; k <= N; ++k)
      for (int f = 0; f < REC; ++f) vrec[qs_blk(b / TL, N, k, REC, b % TL) + (size_t)f * TL] = (qs_real)rec[((size_t)b * (N + 1) + k) * REC + f];
  QsBufs q{vrec.data(), {it0.data(), it1.data()}, st.data(), st2.data(), sb.data(), prod.data(), res.data(), stp.data(), pd.data(), pi32.data(), N, 0};
  Backend bk{*P, q, B, T, N, x0, r, act, xt, ut, status, qp_iter, qp_status, qp_res};
  if (graph) { qs_graph_drive(bk); return bk.n_body; }
  return qs_drive(&bk, 1, 0);
}
