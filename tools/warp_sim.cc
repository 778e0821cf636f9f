// tools/warp_sim.cc -- DEVELOPMENT TOOL (not product, not a test): a CPU model of how one warp of the fused
// playout kernel spends its iterations.  32 persistent lanes play real games with the product's rules header
// compiled for the host; per iteration the model records which of the kernel's branch regions (MOVE, FLOOD)
// execute and with how many active lanes, and prices an iteration with the SASS instruction counts measured
// on the GPU (profiles/r1_playout_v18_regions.txt: MOVE 435, FLOOD 122, loop + refresh + rare ~63).  It is
// used to compare SCHEDULING policies before spending GPU time on them:
//   policy 0  the round-1 kernel: a lane that owes flood visits does not move
//   policy 1  colour overlap: the flood of colour c only touches flag bits of c's pegs and the opponent's
//             move only reads its own pegs' flags, so the opponent moves while c's flood is still running
//   policy 2  policy 1 + the FLOOD region runs twice in iterations where at least T lanes owe visits
//   policy 3  policy 1 + MOVE is skipped in iterations where fewer than T lanes are ready to move
//   policy 4  policy 1 + the FLOOD region only runs every T-th iteration (visits are batched)
//   policy 6  policy 1 + a second FLOOD pass, only for lanes whose next move is blocked by the flood, when >= T are
//   policy 5  policy 1 + the FLOOD region only runs when at least T lanes owe a visit, or one has waited 3 iterations
// Work lists (compile time): the entry stack of flood_visit_entry (default), -DSIM_FRONTIER (one frontier word per
// column) or -DSIM_COLUMNS (the kernel's: a set of columns, flood_visit_columns; "stack depth" = columns in the set).
// Build: g++ -O2 -std=c++17 -I twixt_for_open_spiel_b200/csrc -o /tmp/warp_sim tools/warp_sim.cc
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "twixt_engine.cuh"
#include "twixt_philox.cuh"

using namespace twixt;

struct CachedRec : public RecordRef<1> {
  uint32_t cache[6];
  static constexpr bool kCountCache = true;
  uint32_t cache_ld(int i) const { return cache[i]; }
  void cache_st(int i, uint32_t v) { cache[i] = v; }
  void note_peg(int x, int y, int delta) {
    const uint32_t inc = (1u | ((y == 0 || y == n() - 1) ? 32u : 0u)) << (8 * (x & 3));
    cache[x >> 2] = delta > 0 ? cache[x >> 2] + inc : cache[x >> 2] - inc;
  }
};

// A flood work list that MERGES entries of the same column: one frontier word per board column + a dirty mask.
// Drop-in for the stack interface used by flood_visit_entry.
struct FrontierStack {
  uint32_t f[24];
  uint32_t dirty = 0;
  int sp = 0;  // number of dirty columns (for the depth histogram)
  bool overflow = false;
  FrontierStack() { for (auto& w : f) w = 0; }
  bool empty() const { return dirty == 0; }
  void push(uint32_t e) {
    const int c = static_cast<int>(e >> 24);
    f[c] |= e & 0xFFFFFFu;
    dirty |= 1u << c;
    sp = __builtin_popcount(dirty);
  }
  void push4_if(const bool c[4], const uint32_t e[4]) {
    for (int i = 0; i < 4; ++i) if (c[i]) push(e[i]);
  }
  uint32_t top() const {
    const int c = __builtin_ctz(dirty);
    return (static_cast<uint32_t>(c) << 24) | f[c];
  }
  void pop() {
    const int c = __builtin_ctz(dirty);
    f[c] = 0;
    dirty &= dirty - 1;
    sp = __builtin_popcount(dirty);
  }
};
// The set of columns still to expand (flood_visit_columns): no entries at all, so the visits are made below.
struct ColumnSet {
  uint32_t todo = 0;
  int sp = 0;
  bool empty() const { return todo == 0u; }
};
#if defined(SIM_COLUMNS)
using SimStack = ColumnSet;
#elif defined(SIM_FRONTIER)
using SimStack = FrontierStack;
#else
using SimStack = LocalStack<64>;
#endif

struct Lane {
  std::vector<uint32_t> rec;
  CachedRec b;
  Header h;
  SimStack stk;
  uint32_t pendc[2] = {0, 0}, originc[2] = {0, 0};
  int run_colour = 0, fplane = P_START;
  bool playing = false, have = false;
  int sx = 0, sy = 0, step = 0;
  uint64_t stream = 0;
  bool swap_next = false;
  int load_wait = 0;
};

static uint32_t word_for(uint64_t seed, uint64_t stream, int step) {
  uint32_t r[4];
  philox4x32_10(static_cast<uint32_t>(stream), static_cast<uint32_t>(stream >> 32), static_cast<uint32_t>(step) >> 2, 0u,
                static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), r);
  return r[step & 3];
}

int main(int argc, char** argv) {
  const int n = argc > 1 ? atoi(argv[1]) : 24;
  const int policy = argc > 2 ? atoi(argv[2]) : 0;
  const int thresh = argc > 3 ? atoi(argv[3]) : 8;
  const int games_per_lane = argc > 4 ? atoi(argv[4]) : 6;
  const int warps = argc > 5 ? atoi(argv[5]) : 8;
  const double c_move = 435, c_flood = 122, c_loop = 63;
  const uint64_t seed = 0x7477697854ull;
  double cost = 0;
  long iters = 0, it_move = 0, it_flood = 0, lanes_move = 0, lanes_flood = 0, plies = 0, floods = 0, visits = 0;
  long hist[16] = {0};
  long depth_hist[66] = {0};
  for (int w = 0; w < warps; ++w) {
    std::vector<Lane> L(32);
    int next_game[32];
    for (int l = 0; l < 32; ++l) next_game[l] = 0;
    auto take = [&](int l) {
      Lane& a = L[l];
      if (next_game[l] >= games_per_lane) { a.have = false; return; }
      a.rec.assign(record_words(n), 0u);
      a.b.p = a.rec.data();
      a.b.n_rt = n;
      init_record(a.b);
      load_header(a.b, a.h);
      count_cache_build(a.b);
      a.stream = (static_cast<uint64_t>(w) * 32 + l) * 1000 + next_game[l]++;
      a.step = 0;
      a.playing = true;
      a.have = true;
      a.pendc[0] = a.pendc[1] = 0;
      a.stk = SimStack();
      select_legal(a.b, a.h, static_cast<int>(playout_index(word_for(seed, a.stream, 0), legal_count(a.h, n))), a.sx, a.sy);
      a.swap_next = false;
      a.load_wait = 1;
    };
    for (int l = 0; l < 32; ++l) take(l);
    long cur_visits[32] = {0};
    for (;;) {
      bool any = false;
      for (int l = 0; l < 32; ++l) any |= L[l].have;
      if (!any) break;
      ++iters;
      double c = c_loop;
      // RARE
      for (int l = 0; l < 32; ++l) {
        Lane& a = L[l];
        if (!a.have) continue;
        if (a.load_wait > 0) { --a.load_wait; continue; }
        const bool flood_busy = !a.stk.empty() || a.pendc[0] || a.pendc[1];
        if (!a.playing && !flood_busy) take(l);
        if (a.have && a.swap_next) { swap_first_move(a.b, a.h, a.sx, a.sy); a.swap_next = false; }
      }
      // who can move
      bool ready[32];
      int nready = 0;
      for (int l = 0; l < 32; ++l) {
        Lane& a = L[l];
        ready[l] = false;
        if (!a.have || a.load_wait > 0 || !a.playing) continue;
        const int mover = static_cast<int>(a.h.ply & 1u);
        if (policy == 0) ready[l] = a.stk.empty() && !a.pendc[0] && !a.pendc[1];
        else ready[l] = a.pendc[mover] == 0u && !(!a.stk.empty() && a.run_colour == mover);
        nready += ready[l];
      }
      int nowing = 0;
      for (int l = 0; l < 32; ++l) nowing += L[l].have && (!L[l].stk.empty() || L[l].pendc[0] || L[l].pendc[1]);
      // (policy 3 only waits for lanes that a flood-only iteration can actually free)
      const bool do_move = nready > 0 && !(policy == 3 && nready < thresh && nowing > 0 && nready + nowing >= thresh);
      if (do_move) {
        ++it_move;
        c += c_move;
        for (int l = 0; l < 32; ++l) {
          if (!ready[l]) continue;
          Lane& a = L[l];
          ++lanes_move;
          ++plies;
          const Placement pl = begin_move<true>(a.b, a.h, a.sx, a.sy);
          uint32_t pend = 0;
          const bool win = link_move<true>(a.b, pl, pend);
          finish_move(a.h, pl, win);
          a.pendc[pl.player] = pend;
          a.originc[pl.player] = flood_entry(pl.x, 1u << pl.y);
          if (pend) { ++floods; }
          ++a.step;
          a.playing = a.h.result == kOpen;
          if (a.playing) {
            select_legal(a.b, a.h, static_cast<int>(playout_index(word_for(seed, a.stream, a.step), legal_count(a.h, n))), a.sx, a.sy);
            a.swap_next = is_swap(a.h, static_cast<uint32_t>(a.sx * n + a.sy));
          }
        }
      }
      // FLOOD (possibly twice)
      int passes = 1;
      if (policy == 4 && (iters % thresh) != 0) passes = 0;
      if (policy == 5) {
        int owing = 0;
        static long waited = 0;
        for (int l = 0; l < 32; ++l) owing += L[l].have && (!L[l].stk.empty() || L[l].pendc[0] || L[l].pendc[1]);
        if (owing == 0) waited = 0;
        else if (owing < thresh && waited < 2) { passes = 0; ++waited; }
        else waited = 0;
      }
      if (policy == 2) {
        int owing = 0;
        for (int l = 0; l < 32; ++l) owing += L[l].have && (!L[l].stk.empty() || L[l].pendc[0] || L[l].pendc[1]);
        if (owing >= thresh) passes = 2;
      }
      if (policy == 6) {
        int blocked = 0;
        for (int l = 0; l < 32; ++l) {
          Lane& a = L[l];
          if (!a.have || a.load_wait > 0) continue;
          const int mover = static_cast<int>(a.h.ply & 1u);
          const bool blk = a.pendc[mover] != 0u || (!a.stk.empty() && a.run_colour == mover);
          blocked += blk;
        }
        if (blocked >= thresh) passes = 2;
      }
      for (int p = 0; p < passes; ++p) {
        int nf = 0;
        for (int l = 0; l < 32; ++l) {
          Lane& a = L[l];
          if (!a.have || !(!a.stk.empty() || a.pendc[0] || a.pendc[1])) continue;
          if (policy == 6 && p == 1) {  // second pass: only lanes whose next move waits for the flood
            const int mover = static_cast<int>(a.h.ply & 1u);
            if (!(a.pendc[mover] != 0u || (!a.stk.empty() && a.run_colour == mover))) continue;
          }
          ++nf;
          ++visits;
          uint32_t e = 0;
          if (a.stk.empty()) {
            // begin the flood that blocks the sooner move: the colour to move next first
            const int mover = static_cast<int>(a.h.ply & 1u);
            const int col = a.pendc[mover] ? mover : 1 - mover;
            const bool start = (a.pendc[col] & kFloodStart) != 0u;
            a.fplane = start ? P_START : P_END;
            a.pendc[col] &= start ? ~kFloodStart : ~kFloodEnd;
            a.run_colour = col;
            e = a.originc[col];
#if defined(SIM_COLUMNS)
            a.stk.todo = 1u << (e >> 24);
#endif
          } else {
#if !defined(SIM_COLUMNS)
            e = a.stk.top();
            a.stk.pop();
#endif
          }
#if defined(SIM_COLUMNS)
          flood_visit_columns(a.b, a.run_colour == kRed ? P_RED : P_BLUE, a.fplane, a.stk.todo);
          a.stk.sp = __builtin_popcount(a.stk.todo);
#else
          flood_visit_entry(a.b, a.fplane, a.stk, e);
#endif
          depth_hist[a.stk.sp]++;
          ++cur_visits[l];
          if (a.stk.empty()) {
            hist[cur_visits[l] < 15 ? cur_visits[l] : 15]++;
            cur_visits[l] = 0;
          }
        }
        if (nf > 0) { ++it_flood; c += c_flood; lanes_flood += nf; }
      }
      cost += c;
    }
  }
  printf("n=%d policy=%d T=%d  plies=%ld iters=%ld  MOVE: %ld iters, %.2f lanes  FLOOD: %ld passes, %.2f lanes\n", n, policy,
         thresh, plies, iters, it_move, double(lanes_move) / it_move, it_flood, double(lanes_flood) / it_flood);
  printf("  floods/move=%.3f visits/move=%.3f  model cost/ply=%.1f warp-instr/32 lanes -> %.2f thread-slots per ply\n",
         double(floods) / plies, double(visits) / plies, cost / plies * 1.0, cost * 32 / plies);
  printf("  visits-per-flood(plane) histogram:");
  for (int i = 1; i < 16; ++i) printf(" %d:%ld", i, hist[i]);
  printf("\n  stack depth after a visit (entries): ");
  long tot = 0, acc = 0;
  for (int i = 0; i < 66; ++i) tot += depth_hist[i];
  for (int i = 0; i < 66; ++i) {
    acc += depth_hist[i];
    if (depth_hist[i]) printf(" %d:%.5f", i, 1.0 - double(acc) / tot);
  }
  printf("\n");
  return 0;
}
