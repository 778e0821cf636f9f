// TEST-ONLY: the blocked-plane derivation of the fused playout (derive_blocked_word in
// twixt_for_open_spiel_b200/csrc/twixt_engine.cuh, run by derive_blocked_kernel after the playout kernel)
// on the HOST, next to the per-move rule of host_engine_harness.cc, so that `pytest -m "not gpu"` can check
// that the two agree.  Never part of libtwixt_b200.so.
#include "host_engine_harness.cc"

namespace {

// The playout kernel's accessor with the blocked plane left alone, as link_move<true, false> leaves it.
struct NoBlockedSmemRec : SmemRec {
  void or_blocked3(int, const uint32_t*) {}
};

// derive_blocked_kernel's work for one record: mode = min(starting ply, 2), occ = the cells occupied at the
// start (read for mode 2 only).  Mode 0 stores the derived plane, the others OR it in.
void derive_pass(uint32_t* rec, int n, uint32_t mode, const uint32_t* occ) {
  Rec b{rec, n};
  uint32_t out[32];
  for (int x = 0; x < n; ++x) {
    const uint32_t o0 = mode == 2u ? occ[x] : 0u;
    const uint32_t o1 = mode == 2u && x + 1 < n ? occ[x + 1] : 0u, o2 = mode == 2u && x + 2 < n ? occ[x + 2] : 0u;
    const uint32_t link[4] = {b.ld(P_LINK0 + 0, x), b.ld(P_LINK0 + 1, x), b.ld(P_LINK0 + 2, x), b.ld(P_LINK0 + 3, x)};
    uint32_t bits = 0u;
    for (int c = P_RED; c <= P_BLUE; ++c) {
      const uint32_t p0 = b.ld(c, x), p1 = b.ld_guard(c, x + 1), p2 = b.ld_guard(c, x + 2);
      bits |= derive_blocked_word(p0, p1, p2, p0 & ~o0, p1 & ~o1, p2 & ~o2, link);
    }
    out[x] = (mode != 0u ? b.ld(P_BLOCKED, x) : 0u) | bits;
  }
  for (int x = 0; x < n; ++x) b.st(P_BLOCKED, x, out[x]);
}

}  // namespace

extern "C" {

// the derived plane of the position in `rec` (every peg counted as placed since the plane was empty)
void bh_derive_blocked(const uint32_t* rec, int n, uint32_t* out) {
  std::vector<uint32_t> tmp(rec, rec + record_words(n));
  derive_pass(tmp.data(), n, 0u, nullptr);
  for (int x = 0; x < n; ++x) out[x] = tmp[kHeaderWords + P_BLOCKED * n + x];
}

// he_playout_smem without the per-move blocked bookkeeping, followed by the derivation pass: what the fused
// playout kernel and derive_blocked_kernel together do to one env
int bh_playout_derived(uint32_t* rec, int n, uint64_t seed, uint64_t stream, int max_plies, int64_t* actions_out) {
  Rec r{rec, n};
  Header h;
  load_header(r, h);
  const uint32_t mode = h.ply < 2u ? h.ply : 2u;
  std::vector<uint32_t> occ(n);
  for (int x = 0; x < n; ++x) occ[x] = r.ld(P_RED, x) | r.ld(P_BLUE, x);
  NoBlockedSmemRec b;
  b.take(rec, n);
  const int steps = playout_like_kernel(b, h, n, seed, stream, max_plies, actions_out);
  b.give(rec);
  store_header(r, h);
  derive_pass(rec, n, mode, occ.data());
  return steps;
}

}  // extern "C"
