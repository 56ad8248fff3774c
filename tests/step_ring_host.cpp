// TEST HARNESS -- host build of qs_step (safe_mpc_b200/csrc/qp_split.cuh) with its two operand sources: QsStepGlobal (global memory,
// the thread form) and HostStepRing, the host stand-in of the ring of the staged step kernels (qp.cu: StepRing) -- the same chunk table
// (qs_sp) and slot layout, filled by memcpy.  Every read of the ring checks that its chunk is held (acquired, not yet released) and that
// the field lies in it; chunks are acquired in order, a slot is refilled only after its chunk was released, and a released or skipped
// slot is overwritten with NaN.  Not part of the product.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../safe_mpc_b200/csrc/qp_split.cuh"

using namespace smpc;

namespace {
int g_errors = 0;

struct HostStepRing {
  static constexpr int NS = 3;
  const QsBufs& q;
  size_t blk;
  int kk, mode, ln;
  StageFlags F;
  std::vector<unsigned char> sm;
  int slot_chunk[NS] = {-1, -1, -1};
  int acquired = -1;
  bool released[QSC_N] = {};
  HostStepRing(const smpc_problem_t& P, const QsBufs& q_, int tile, int lane, int k, int kk_, int mode_)
      : q(q_), blk((size_t)tile * (q_.N + 1) + k), kk(kk_), mode(mode_), ln(lane), F(qs_flags(P, k)), sm((size_t)NS * qs_chunk_max_bytes(), 0xff) {
    for (int c = 0; c < NS; ++c) issue(c);
  }
  const void* gsrc(const QsPiece& p) const {
    switch (p.a) {
      case QA_IT: return q.it[kk & 1] + (blk * NIT + p.f0) * TL;
      case QA_ST: return q.st + (blk * NIT + p.f0) * TL;
      case QA_ST2: return q.st2 + (blk * NS2 + p.f0) * TL;
      case QA_REC: return q.rec + (blk * REC + p.f0) * TL;
      default: return q.prod + (blk * NPROD + p.f0) * TL;
    }
  }
  void issue(int c) {
    if (c >= QSC_N) return;
    const int s = c % NS;
    if (slot_chunk[s] >= 0 && !released[slot_chunk[s]]) ++g_errors;
    unsigned char* dst = sm.data() + (size_t)s * qs_chunk_max_bytes();
    std::memset(dst, 0xff, qs_chunk_max_bytes());
    slot_chunk[s] = c;
    if (!qs_chunk_on(c, F)) return;
    if (qs_chunk_bytes(mode, c) > qs_chunk_max_bytes()) ++g_errors;
    for (int i = 0; i < QSC_PIECES; ++i) {
      const QsPiece p = qs_sp(mode, c, i);
      if (p.n == 0) continue;
      if (qs_sp_bytes(p) % 16) ++g_errors;               // (bulk-copy sizes are multiples of 16 bytes)
      std::memcpy(dst, gsrc(p), qs_sp_bytes(p));
      dst += qs_sp_bytes(p);
    }
  }
  void acquire(int c) {
    if (c != acquired + 1 || slot_chunk[c % NS] != c) ++g_errors;
    acquired = c;
  }
  void release(int c) {
    if (c > acquired || released[c]) ++g_errors;
    released[c] = true;
    std::memset(sm.data() + (size_t)(c % NS) * qs_chunk_max_bytes(), 0xff, qs_chunk_max_bytes());
    issue(c + NS);
  }
  template <class T> double ld(int c, int a, int f) const {
    const int off = qs_chunk_off(mode, c, a, f);
    if (off < 0 || c > acquired || released[c] || !qs_chunk_on(c, F) || slot_chunk[c % NS] != c) { ++g_errors; return std::nan(""); }
    T v;
    std::memcpy(&v, sm.data() + (size_t)(c % NS) * qs_chunk_max_bytes() + off + ln * sizeof(T), sizeof(T));
    return (double)v;
  }
  double it(int c, int f) const { return ld<double>(c, QA_IT, f); }
  double st(int c, int f) const { return ld<qs_real>(c, QA_ST, f); }
  double st2(int c, int f) const { return ld<qs_real>(c, QA_ST2, f); }
  double prod(int c, int f) const { return ld<qs_real>(c, QA_PROD, f); }
  double rec(int c, int f) const { return ld<qs_real>(c, QA_REC, f); }
};

// every array of the solver state of T tiles
struct State {
  std::vector<qs_real> rec, st, st2, sb, prod;
  std::vector<double> it0, it1, res, stp, pd;
  std::vector<int32_t> pi;
  QsBufs q;
  State(int T, int N) {
    const size_t S = (size_t)T * (N + 1) * TL;
    rec.assign(S * REC, 0); st.assign(S * NIT, 0); st2.assign(S * NS2, 0); sb.assign(S * NSB, 0); prod.assign(S * NPROD, 0);
    it0.assign(S * NIT, 0); it1.assign(S * NIT, 0); res.assign(S * NRES, 0); stp.assign(S * NSTP, 0); pd.assign((size_t)T * NPD * TL, 0);
    pi.assign((size_t)T * NPI * TL, 0);
    bind(N);
  }
  State(const State& o) : rec(o.rec), st(o.st), st2(o.st2), sb(o.sb), prod(o.prod), it0(o.it0), it1(o.it1), res(o.res), stp(o.stp), pd(o.pd), pi(o.pi) { bind(o.q.N); }
  void bind(int N) { q = QsBufs{rec.data(), {it0.data(), it1.data()}, st.data(), st2.data(), sb.data(), prod.data(), res.data(), stp.data(), pd.data(), pi.data(), N, 0}; }
};

template <class V> bool same(const V& a, const V& b) { return a.size() == b.size() && std::memcmp(a.data(), b.data(), a.size() * sizeof(a[0])) == 0; }
}  // namespace

// Runs qs_step in every mode on T tiles of seeded random stage blocks, once per operand source, and compares every array bit for bit.
// Returns the number of (kk, mode) runs whose outputs differ; *ring_errors: violations of the ring protocol.
extern "C" int step_ring_check(const smpc_problem_t* P, int T, uint64_t seed, int* ring_errors) {
  const int N = P->N;
  State s0(T, N);
  uint64_t x = seed * 2862933555777941757ull + 3037000493ull;
  auto rnd = [&]() { x = x * 6364136223846793005ull + 1442695040888963407ull; return (double)(x >> 11) * (1.0 / 9007199254740992.0); };
  for (auto& v : s0.rec) v = (qs_real)(rnd() * 2.0 - 1.0);
  for (auto* a : {&s0.st, &s0.st2, &s0.prod}) for (auto& v : *a) v = (qs_real)(rnd() * 2.0 - 1.0);
  for (auto* a : {&s0.it0, &s0.it1}) for (auto& v : *a) v = 0.05 + rnd();       // positive multipliers and slacks
  for (auto& v : s0.pd) v = rnd();
  for (int t = 0; t < T; ++t)
    for (int l = 0; l < TL; ++l) {
      int32_t* pi = s0.pi.data() + qs_pb(t, NPI, l);
      QF(pi, J_ACT) = (l % 7) != 3;                                             // some idle lanes in every warp
      QF(pi, J_REDO) = (l + t) % 3 == 0;
      QF(pi, J_R) = (int)(rnd() * N);
      QF(pi, J_NC) = 1;
    }
  g_errors = 0;
  int bad = 0;
  for (int kk = 0; kk < 2; ++kk)
    for (int mode = 0; mode < 3; ++mode) {
      State a(s0), b(s0);
      for (int t = 0; t < T; ++t)
        for (int k = 0; k <= N; ++k)
          for (int l = 0; l < TL; ++l) {
            qs_step(*P, a.q, t, l, k, kk, mode);
            HostStepRing src(*P, b.q, t, l, k, kk, mode);
            qs_step(*P, b.q, t, l, k, kk, mode, src);
          }
      if (!(same(a.st, b.st) && same(a.prod, b.prod) && same(a.sb, b.sb) && same(a.stp, b.stp) && same(a.st2, b.st2) && same(a.it0, b.it0) &&
            same(a.it1, b.it1)))
        ++bad;
    }
  *ring_errors = g_errors;
  return bad;
}
