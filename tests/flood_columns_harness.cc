// TEST-ONLY: the fused playout kernel's loop (twixt_kernel_playout.cu) compiled for the HOST, on the kernel's
// shared-memory layout of 8n + 4 words per env, with its border-flag flood driven by a set of columns
// (flood_visit_columns in twixt_for_open_spiel_b200/csrc/twixt_engine.cuh).  The same loop can run the flood
// from the entry stack of flood_visit_entry instead, so that tests can compare the number of flood visits
// the two work lists take.  Never part of libtwixt_b200.so.
#include <cstdint>
#include <cstdlib>
#include <vector>

#include "twixt_engine.cuh"
#include "twixt_philox.cuh"

using namespace twixt;

namespace {

const uint8_t* host_select_lut() {
  static uint8_t lut[8 * 256];
  static bool ready = false;
  if (!ready) {
    for (int e = 0; e < 8 * 256; ++e) fill_select_lut(lut, e);
    ready = true;
  }
  return lut;
}

// The kernel's layout (PlayoutRef): planes BLUE, RED, links, START, END, then the 4 pad words, which are
// poisoned; reads of the link window and of the flags carry no bounds test, and any access outside the
// 8n + 4 words of the env aborts.
struct PadRec {
  static constexpr bool kSelectLut = true;
  static constexpr bool kCountCache = true;
  const uint8_t* select_lut() const { return host_select_lut(); }
  std::vector<uint32_t> w;
  uint32_t* blocked;  // the record's blocked plane (global memory in the kernel)
  int n_rt;
  uint32_t cache[6];
  int n() const { return n_rt; }
  int smem_word(int i) const { return i < n_rt ? i + n_rt : (i < 2 * n_rt ? i - n_rt : i); }
  void take(const uint32_t* rec, int n) {
    n_rt = n;
    w.assign(8 * n + 4, 0xDEADBEEFu);
    for (int i = 0; i < 8 * n; ++i) w[smem_word(i)] = rec[kHeaderWords + i];
  }
  void give(uint32_t* rec) const {
    for (int i = 0; i < 8 * n_rt; ++i) rec[kHeaderWords + i] = w[smem_word(i)];
  }
  uint32_t& at(int plane, int col) {
    const int i = plane * n_rt + col;
    if (i < 0 || i >= static_cast<int>(w.size())) std::abort();
    return w[i];
  }
  uint32_t ld(int plane, int col) const { return const_cast<PadRec*>(this)->at(plane, col); }
  void st(int plane, int col, uint32_t v) { at(plane, col) = v; }
  void st_if(bool c, int plane, int col, uint32_t v) {
    if (c) {
      if (col < 0 || col >= n_rt) std::abort();
      st(plane, col, v);
    }
  }
  uint32_t ld_guard(int plane, int col) const {
    return (static_cast<unsigned>(col) < static_cast<unsigned>(n_rt)) ? ld(plane, col) : 0u;
  }
  uint32_t ld_link(int plane, int col) const { return ld(plane, col); }
  uint32_t ld_any(int plane, int col) const { return ld(plane, col); }
  uint32_t ld_pegs(int plane, int col) const { return ld(plane ^ 1, col); }
  void st_pegs(int plane, int col, uint32_t v) { st(plane ^ 1, col, v); }
  uint32_t ld_pegs_guard(int plane, int col) const { return ld_guard(plane ^ 1, col); }
  void or_blocked3(int x, const uint32_t blk[3]) {
    blocked[x] |= blk[0];
    blocked[x - 1 > 0 ? x - 1 : 0] |= blk[1];
    blocked[x - 2 > 0 ? x - 2 : 0] |= blk[2];
  }
  uint32_t cache_ld(int i) const { return cache[i]; }
  void cache_st(int i, uint32_t v) { cache[i] = v; }
  void note_peg(int x, int y, int delta) {
    const uint32_t inc = (1u | ((y == 0 || y == n() - 1) ? 32u : 0u)) << (8 * (x & 3));
    cache[x >> 2] = delta > 0 ? cache[x >> 2] + inc : cache[x >> 2] - inc;
  }
};

// The kernel's loop for one env: moves interleaved with single flood visits, the opponent moving while a
// colour's flood runs, the lowest owed flood started first, the following move chosen between placement
// and link evaluation, the swap's first half run ahead of the move.  kColumns: the work list is the column
// set `todo` (as in the kernel); otherwise a stack of entries that never overflows.
template <bool kColumns>
int playout(PadRec& b, Header& h, int n, uint64_t seed, uint64_t stream, int max_plies, int64_t* actions_out,
            int64_t* visits) {
  count_cache_build(b);
  const uint32_t s_lo = static_cast<uint32_t>(stream), s_hi = static_cast<uint32_t>(stream >> 32);
  const uint32_t k_lo = static_cast<uint32_t>(seed), k_hi = static_cast<uint32_t>(seed >> 32);
  auto word_at = [&](uint32_t index) {
    uint32_t r[4];
    philox4x32_10(s_lo, s_hi, index >> 2, 0u, k_lo, k_hi, r);
    return r[index & 3u];
  };
  int step = 0;
  uint32_t pend = 0, fcol = 0, todo = 0;
  uint32_t origin[2] = {0u, 0u};  // the newest peg of each colour: its column bit (kColumns) or its stack entry
  int fplane = P_START;
  LocalStack<8 * 24 * 24> stk;  // (one entry per visit at most: cannot overflow)
  auto running = [&]() { return kColumns ? todo != 0u : !stk.empty(); };
  bool playing = h.result == kOpen && max_plies > 0;
  int sx = 0, sy = 0;
  if (playing) select_legal(b, h, static_cast<int>(playout_index(word_at(0), static_cast<uint32_t>(legal_count(h, n)))), sx, sy);
  int sact = sx * n + sy;
  bool swap_next = playing && is_swap(h, static_cast<uint32_t>(sact));
  while (playing || pend != 0u || running()) {
    if (swap_next) {
      swap_first_move(b, h, sx, sy);
      swap_next = false;
    }
    const uint32_t mover = h.ply & 1u;
    const bool flood_blocks = ((pend >> (2u * mover)) & 3u) != 0u || (running() && fcol == mover);
    if (playing && !flood_blocks) {
      if (actions_out) actions_out[step] = sact;
      const Placement pl = begin_move<true>(b, h, sx, sy);
      Header hn = h;
      hn.ply = h.ply + 1u;
      int nx, ny;
      select_legal(b, hn, static_cast<int>(playout_index(word_at(static_cast<uint32_t>(step) + 1u), static_cast<uint32_t>(legal_count(hn, n)))), nx, ny);
      uint32_t owed;
      const bool win = link_move<true>(b, pl, owed);
      finish_move(h, pl, win);
      pend |= owed << (2 * pl.player);
      origin[pl.player] = kColumns ? 1u << pl.x : flood_entry(pl.x, 1u << pl.y);
      ++step;
      playing = h.result == kOpen && step < max_plies;
      sx = nx;
      sy = ny;
      sact = nx * n + ny;
      swap_next = playing && is_swap(h, static_cast<uint32_t>(sact));
    }
    if (running() || pend != 0u) {
      const bool begin = !running();
      const uint32_t lsb = pend & (0u - pend);
      const bool blue = (lsb & 12u) != 0u;
      fplane = begin ? ((lsb & 5u) != 0u ? P_START : P_END) : fplane;
      fcol = begin ? (blue ? 1u : 0u) : fcol;
      pend ^= begin ? lsb : 0u;
      ++*visits;
      if (kColumns) {
        todo = begin ? origin[blue ? 1 : 0] : todo;
        flood_visit_columns(b, fcol == kRed ? P_RED : P_BLUE, fplane, todo);
      } else {
        flood_visit_entry(b, fplane, stk, stk.top_or(origin[blue ? 1 : 0]));
      }
    }
  }
  return step;
}

}  // namespace

extern "C" {

// Plays the env in `rec` (a record as in include/twixt_b200.h) to its end or `max_plies` with the Philox stream
// of the fused playout; returns the plies played, writes the actions and adds the flood visits to *visits.
int fc_playout(uint32_t* rec, int n, uint64_t seed, uint64_t stream, int max_plies, int columns, int64_t* actions_out,
               int64_t* visits) {
  RecordRef<1> r{rec, n};
  Header h;
  load_header(r, h);
  PadRec b;
  b.take(rec, n);
  b.blocked = rec + kHeaderWords + P_BLOCKED * n;
  const int steps = columns ? playout<true>(b, h, n, seed, stream, max_plies, actions_out, visits)
                            : playout<false>(b, h, n, seed, stream, max_plies, actions_out, visits);
  if (b.w[8 * n] != 0xDEADBEEFu || b.w[8 * n + 1] != 0xDEADBEEFu || b.w[8 * n + 2] != 0xDEADBEEFu ||
      b.w[8 * n + 3] != 0xDEADBEEFu)
    std::abort();  // the pad words are read, never written
  b.give(rec);
  store_header(r, h);
  return steps;
}

}  // extern "C"
