// twixt_engine.cuh -- the per-env TwixT rules on the bit-plane state record.
//
// One game ("env") is a record of 4 header words + 9 bit-planes of n column
// words (layout: include/twixt_b200.h).  Everything here is scalar code for
// ONE env, templated on a memory accessor so the same rules run
//   * thread-per-env on the record in global memory      (apply kernel),
//   * thread-per-env on a record staged in shared memory (fused playout),
// and -- compiled for the host by tests/host_engine_harness.cc only -- on a
// plain array, so the rules can be checked against the oracle without a GPU.
// The product library never runs this on the CPU.
//
// Reference semantics reproduced (file:line under
// /root/reference/open_spiel/games/twixt/):
//   legal lists + swap quirk   twixtboard.cc:252-276, 457-493, 633-640
//   peg, links, crossings      twixtboard.cc:501-556, 38-144, 176-190
//   border flags + flood       twixtboard.cc:537-546, 557-588
//   result                     twixtboard.cc:192-207
//   observation planes         twixt.cc:76-132, twixtboard.cc:590-597
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define TW_HD __host__ __device__ __forceinline__
#define TW_HD_NOINLINE __host__ __device__ __noinline__
#else
#define TW_HD inline
#define TW_HD_NOINLINE inline
#endif

namespace twixt {

enum : int { P_RED = 0, P_BLUE = 1, P_LINK0 = 2, P_START = 6, P_END = 7, P_BLOCKED = 8, kNumStatePlanes = 9 };
enum : int { kHeaderWords = 4 };
enum : int { kOpen = 0, kRedWin = 1, kBlueWin = 2, kDraw = 3 };
enum : int { kRed = 0, kBlue = 1 };
enum : int { kTerminalPlayer = -4 };
enum : uint32_t { kNoMove = 0xFFFFFFFFu };

// (Padding records to whole 128-byte lines -- 224 words at n = 24 -- was measured in round 2: no gain for the
// kernels that read only a record's head, because their loads already carry the 64-byte L2 fetch hint, which
// makes any 208-byte head cost four 64-byte granules whatever its offset; DESIGN.md section 9.)
TW_HD int record_words(int n) { return (kHeaderWords + kNumStatePlanes * n + 3) & ~3; }

TW_HD int tw_popc(uint32_t v) {
#if defined(__CUDA_ARCH__)
  return __popc(v);
#else
  return __builtin_popcount(v);
#endif
}
// index of the lowest set bit, v != 0
TW_HD int tw_ctz(uint32_t v) {
#if defined(__CUDA_ARCH__)
  return __ffs(static_cast<int>(v)) - 1;
#else
  return __builtin_ctz(v);
#endif
}
// index of the highest set bit, v != 0 (one FLO on the device; tw_ctz needs a BREV in front of it)
TW_HD int tw_msb(uint32_t v) {
#if defined(__CUDA_ARCH__)
  return 31 - __clz(static_cast<int>(v));
#else
  return 31 - __builtin_clz(v);
#endif
}

TW_HD int tw_min(int a, int b) { return a < b ? a : b; }
TW_HD int tw_max(int a, int b) { return a > b ? a : b; }

// Compass offsets (twixtcell.h:58-68), biased by +2 and packed one nibble per
// direction so a lookup is a shift and a mask.
TW_HD int dir_dx(int d) { return static_cast<int>((0x10013443u >> (4 * d)) & 15u) - 2; }
TW_HD int dir_dy(int d) { return static_cast<int>((0x43100134u >> (4 * d)) & 15u) - 2; }

struct Header {
  uint32_t ply;       // Board::move_counter_
  uint32_t result;    // kOpen..kDraw
  uint32_t swapped;   // 0/1
  uint32_t move_one;  // action of the first move or kNoMove
  int cnt[2];         // empty cells red / blue may play on
};

TW_HD void unpack_header(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, Header& h) {
  h.ply = w0;
  h.result = w1 & 3u;
  h.swapped = (w1 >> 2) & 1u;
  h.move_one = w2;
  h.cnt[0] = static_cast<int>(w3 & 0xFFFFu);
  h.cnt[1] = static_cast<int>(w3 >> 16);
}
TW_HD void pack_header(const Header& h, uint32_t& w0, uint32_t& w1, uint32_t& w2, uint32_t& w3) {
  w0 = h.ply;
  w1 = h.result | (h.swapped << 2);
  w2 = h.move_one;
  w3 = static_cast<uint32_t>(h.cnt[0]) | (static_cast<uint32_t>(h.cnt[1]) << 16);
}

// Accessor over a record whose words are `stride` words apart (1 for a record
// in global memory, the number of threads sharing the staging buffer for a
// record transposed into shared memory).
// kN > 0 fixes the board size at compile time (fused playout), kN == 0 reads it
// from n_rt.
template <int kStride, int kN = 0>
struct RecordRef {
  uint32_t* p;
  int n_rt;
  TW_HD int n() const { return kN > 0 ? kN : n_rt; }
  TW_HD uint32_t word(int w) const { return p[w * kStride]; }
  TW_HD void set_word(int w, uint32_t v) { p[w * kStride] = v; }
  TW_HD uint32_t ld(int plane, int col) const { return p[(kHeaderWords + plane * n() + col) * kStride]; }
  TW_HD void st(int plane, int col, uint32_t v) { p[(kHeaderWords + plane * n() + col) * kStride] = v; }
  // conditional store; `col` may be outside the board when `c` is false
  TW_HD void st_if(bool c, int plane, int col, uint32_t v) {
    if (c) st(plane, col, v);
  }
  // column outside the board reads as empty
  TW_HD uint32_t ld_guard(int plane, int col) const {
    return (static_cast<unsigned>(col) < static_cast<unsigned>(n())) ? ld(plane, col) : 0u;
  }
  // Two relaxed reads for the hot straight-line code, which an accessor may implement WITHOUT a bounds
  // test if its storage allows (the fused playout kernel's shared-memory layout does):
  //  ld_link  link word of column `col` >= -3: must read as empty at column -1; at every other off-board
  //           column the callers only use it for targets that are off the board themselves (link_move:
  //           a target in column x+dx reads west endpoints in x+dx-1 .. x+dx+1 clipped to x-3 .. x+1,
  //           twixt_crossing.inc, so a target on the board never looks left of column -1)
  //  ld_any   word whose value the caller ignores when the column is off the board
  TW_HD uint32_t ld_link(int plane, int col) const { return ld_guard(plane, col); }
  TW_HD uint32_t ld_any(int plane, int col) const { return ld_guard(plane, col); }
  // the two peg planes (P_RED / P_BLUE) are the hot ones: an accessor may keep them
  // in faster memory than the rest, so the rules name them separately
  TW_HD uint32_t ld_pegs(int plane, int col) const { return ld(plane, col); }
  TW_HD void st_pegs(int plane, int col, uint32_t v) { st(plane, col, v); }
  TW_HD uint32_t ld_pegs_guard(int plane, int col) const { return ld_guard(plane, col); }
  // the blocked plane is write-only for the rules (only ObservationTensor reads it)
  TW_HD void or_blocked(int col, uint32_t bits) { st(P_BLOCKED, col, ld(P_BLOCKED, col) | bits); }
  // new blocked-east bits of the columns x, x-1, x-2 (blk[i] for column x-i; all zero most of the time)
  TW_HD void or_blocked3(int x, const uint32_t blk[3]) {
    if (blk[0]) or_blocked(x, blk[0]);
    if (blk[1]) or_blocked(x - 1, blk[1]);
    if (blk[2]) or_blocked(x - 2, blk[2]);
  }
  // no per-column count cache on a plain record (see count_cache_* below), no select table
  static constexpr bool kCountCache = false;
  static constexpr bool kSelectLut = false;
  TW_HD void note_peg(int, int, int) {}
};

// Flood-fill work stack.  An entry names up to 24 cells of ONE column:
// (column << 24) | row mask -- the flood discovers unflagged neighbours column
// by column, so a visit pushes at most four entries instead of eight cells.
TW_HD uint32_t flood_entry(int column, uint32_t row_mask) { return (static_cast<uint32_t>(column) << 24) | row_mask; }

// ... kept in a thread-local array (apply kernel, host tests).
template <int kCap>
struct LocalStack {
  uint32_t v[kCap];
  int sp = 0;
  bool overflow = false;
  TW_HD bool empty() const { return sp == 0; }
  TW_HD void push(uint32_t e) {
    if (sp < kCap) v[sp++] = e;
    else overflow = true;
  }
  TW_HD void push_if(bool c, uint32_t e) {
    if (c) push(e);
  }
  // the (up to) four entries a flood visit discovers; a stack may test for room once for all four
  TW_HD void push4_if(const bool c[4], const uint32_t e[4]) {
    for (int i = 0; i < 4; ++i) push_if(c[i], e[i]);
  }
  TW_HD uint32_t top() const { return v[sp - 1]; }
  TW_HD void pop() { --sp; }
  // pop the top entry, or take `otherwise` if there is none
  TW_HD uint32_t top_or(uint32_t otherwise) { return sp > 0 ? v[--sp] : otherwise; }
};

template <class B>
TW_HD void load_header(const B& b, Header& h) {
  unpack_header(b.word(0), b.word(1), b.word(2), b.word(3), h);
}
template <class B>
TW_HD void store_header(B& b, const Header& h) {
  uint32_t w0, w1, w2, w3;
  pack_header(h, w0, w1, w2, w3);
  b.set_word(0, w0);
  b.set_word(1, w1);
  b.set_word(2, w2);
  b.set_word(3, w3);
}

TW_HD uint32_t full_rows(int n) { return (1u << n) - 1u; }
TW_HD uint32_t inner_rows(int n) { return ((1u << n) - 1u) & ~1u & ~(1u << (n - 1)); }

// Cells `player` may ever play on in column x: red everything in columns
// 1..n-2, blue rows 1..n-2 of every column (InitializeLegalActions,
// twixtboard.cc:252-276; corners are off-board, 625-631).  Written with selects
// only: these helpers sit in the hottest loops and a branch per call costs more
// than computing both sides.
TW_HD uint32_t playable_word(int n, int player, int x) {
  const uint32_t red = (x >= 1 && x <= n - 2) ? full_rows(n) : 0u;
  return player == kRed ? red : inner_rows(n);
}

// The initial record of an env (Board::Board, twixtboard.cc:168-174).
template <class B>
TW_HD void init_record(B& b) {
  int n = b.n();
  int words = record_words(n);
  for (int w = kHeaderWords; w < words; ++w) b.set_word(w, 0u);
  Header h;
  h.ply = 0; h.result = kOpen; h.swapped = 0; h.move_one = kNoMove;
  h.cnt[0] = h.cnt[1] = n * (n - 2);
  store_header(b, h);
}

TW_HD int current_player(const Header& h) {
  return h.result != kOpen ? static_cast<int>(kTerminalPlayer) : static_cast<int>(h.ply & 1u);
}

// |LegalActions()| (twixt.h:86-90).  At ply 1 blue's list is still the initial
// one -- the occupied first-move cell stays in it as the swap offer
// (twixtboard.cc:485-488) -- from ply 2 on both lists are "playable and empty".
TW_HD int legal_count(const Header& h, int n) {
  const int by_count = (h.ply & 1u) ? h.cnt[kBlue] : h.cnt[kRed];  // (a run-time index would push the header into local memory)
  const int open_count = h.ply == 1u ? n * (n - 2) : by_count;
  return h.result != kOpen ? 0 : open_count;
}

// Legal cells of the player to move in column x (result must be open).
template <class B>
TW_HD uint32_t legal_word(const B& b, const Header& h, int x) {
  const int player = static_cast<int>(h.ply & 1u);
  const uint32_t play = playable_word(b.n(), player, x);
  const uint32_t occ = b.ld_pegs(P_RED, x) | b.ld_pegs(P_BLUE, x);
  return h.ply == 1u ? play : (play & ~occ);
}

// ... of a column that is known to hold a legal cell of the player to move (it was picked from the per-column
// counts, which are zero for red's two forbidden columns): the edge-column test of playable_word is moot
template <class B>
TW_HD uint32_t legal_word_selected(const B& b, const Header& h, int x) {
  const uint32_t play = (h.ply & 1u) == kRed ? full_rows(b.n()) : inner_rows(b.n());
  const uint32_t occ = b.ld_pegs(P_RED, x) | b.ld_pegs(P_BLUE, x);
  return h.ply == 1u ? play : (play & ~occ);
}

template <class B>
TW_HD bool is_legal(const B& b, const Header& h, int action) {
  int n = b.n();
  if (h.result != kOpen) return false;
  if (action < 0 || action >= n * n) return false;
  int x = action / n, y = action - x * n;
  return (legal_word(b, h, x) >> y) & 1u;
}

// The link words a move can touch: the four link planes over the columns
// x-3 .. x+1 around the new peg at column x (index c = column - x + 3).  They
// are fetched once, with independent loads, before the eight directions are
// examined, so the crossing tests themselves run out of registers.
struct LinkWindow {
  uint32_t w[4][5];
};

// How the link window is aligned to the new peg's row.  TW_ALIGN_MUL = 0: (word << 5) >> y, row y+oy at bit
// oy+5 -- two shifts per word on the integer-ALU pipe, the busiest pipe of the playout kernel (74 %).
// TW_ALIGN_MUL = 1: word * 2^(28-y), row y+oy at bit oy+28 -- ONE multiply per word, which issues on the FMA
// pipe (13 % busy); rows above y+3 leave the word at the top, rows below y-2 stay in the low bits where no
// crossing mask looks (the masks of twixt_crossing.inc cover oy = -2 .. +3, i.e. bits 26 .. 31 here).
#ifndef TW_ALIGN_MUL
#define TW_ALIGN_MUL 1
#endif
enum : int { kAlignShift = TW_ALIGN_MUL ? 23 : 0 };

TW_HD uint32_t align_factor(int y) { return TW_ALIGN_MUL ? (1u << (28 - y)) : static_cast<uint32_t>(y); }
TW_HD uint32_t align_word(uint32_t w, uint32_t factor) {
#if TW_ALIGN_MUL
#if defined(__CUDA_ARCH__)
  uint32_t r;  // (inline PTX: the optimiser would turn a multiply by 1 << s back into a shift)
  asm("mul.lo.u32 %0, %1, %2;" : "=r"(r) : "r"(w), "r"(factor));
  return r;
#else
  return w * factor;
#endif
#else
  return (w << 5) >> factor;
#endif
}

// Would the link from the new peg (x, y) in Compass direction d be crossed by
// an existing link, of either colour (twixtboard.cc:519-527 tests HasLink
// only)?  `ly` is the window with every word aligned to the peg's row (see
// above), so that each of the 5..7 tests of a direction is one AND with a
// constant (twixt_crossing.inc, masks written for row y+oy at bit oy+5).
TW_HD bool crossing_blocked(const LinkWindow& ly, int d) {
#define TW_X(plane, c, mask) (ly.w[plane][c] & (static_cast<uint32_t>(mask) << kAlignShift))
#define TW_CROSS_CASE(dir, expr) \
  case dir:                      \
    return (expr) != 0u;
  switch (d) {
#include "twixt_crossing.inc"
  }
#undef TW_CROSS_CASE
#undef TW_X
  return false;
}

// Cell::links_ of (x,y) reassembled from the four west-endpoint planes.
template <class B>
TW_HD uint32_t links_of(const B& b, int x, int y) {
  uint32_t m = 0;
  m |= ((b.ld(P_LINK0 + 0, x) >> y) & 1u) << 0;
  m |= ((b.ld(P_LINK0 + 1, x) >> y) & 1u) << 1;
  m |= ((b.ld(P_LINK0 + 2, x) >> y) & 1u) << 2;
  m |= ((b.ld(P_LINK0 + 3, x) >> y) & 1u) << 3;
  m |= (((b.ld_guard(P_LINK0 + 0, x - 1) << 2) >> y) & 1u) << 4;  // SSW: NNE link of (x-1,y-2)
  m |= (((b.ld_guard(P_LINK0 + 1, x - 2) << 1) >> y) & 1u) << 5;  // WSW: ENE link of (x-2,y-1)
  m |= ((b.ld_guard(P_LINK0 + 2, x - 2) >> (y + 1)) & 1u) << 6;   // WNW: ESE link of (x-2,y+1)
  m |= ((b.ld_guard(P_LINK0 + 3, x - 1) >> (y + 2)) & 1u) << 7;   // NNW: SSE link of (x-1,y+2)
  return m;
}

// ExploreLocalGraph (twixtboard.cc:573-588) gives a border flag to every cell
// reachable from the new peg through links over cells that lack it.  It is
// split into single VISITS so that the fused playout kernel can interleave the
// visits of one env with the moves of the other envs of its warp instead of
// making 31 lanes wait for one lane's whole flood.
//
// One visit: pop an ENTRY -- all its cells of one column at once -- and flag +
// push every linked neighbour that lacks the flag.  Word-parallel and
// straight-line: for each of the four neighbour COLUMNS the linked neighbour
// cells are formed directly as a row mask from the link words -- the east
// links are bits of this column's own link words (at the entry's rows) moved
// to their target rows, the west links are bits of the neighbour column's link
// words sitting AT the target rows -- then masked with the flag word.  A row
// shifted off the board meets no link bit.  (Eight data-dependent branches per
// visit cost more than they skipped, and the per-direction formulation was
// 40 % more instructions.)
//
// flood_flag_neighbours is that step for the cells `rows` of column cx: it flags their linked neighbours and
// returns the newly flagged rows of the columns cx+1, cx+2, cx-1, cx-2 in fresh[0..3].
template <class B>
TW_HD void flood_flag_neighbours(B& b, int flag_plane, int cx, uint32_t rows, uint32_t fresh[4]) {
  // links stored at these cells (they are their west endpoints): NNE, ENE, ESE, SSE
  const uint32_t own0 = b.ld(P_LINK0 + 0, cx) & rows, own1 = b.ld(P_LINK0 + 1, cx) & rows;
  const uint32_t own2 = b.ld(P_LINK0 + 2, cx) & rows, own3 = b.ld(P_LINK0 + 3, cx) & rows;
  // linked neighbours per column, as row masks
  const uint32_t e1 = (own0 << 2) | (own3 >> 2);                       // (cx+1, cy+2) NNE, (cx+1, cy-2) SSE
  const uint32_t e2 = (own1 << 1) | (own2 >> 1);                       // (cx+2, cy+1) ENE, (cx+2, cy-1) ESE
  const uint32_t w1 = (b.ld_link(P_LINK0 + 0, cx - 1) & (rows >> 2)) |    // NNE links of (cx-1, cy-2)
                      (b.ld_link(P_LINK0 + 3, cx - 1) & (rows << 2));     // SSE links of (cx-1, cy+2)
  const uint32_t w2 = (b.ld_guard(P_LINK0 + 1, cx - 2) & (rows >> 1)) |   // ENE links of (cx-2, cy-1)
                      (b.ld_guard(P_LINK0 + 2, cx - 2) & (rows << 1));    // ESE links of (cx-2, cy+1)
  // a neighbour column off the board has no linked cells (e1 .. w2 are empty there): its flag word is ignored
  const uint32_t f_e1 = b.ld_any(flag_plane, cx + 1), f_e2 = b.ld_any(flag_plane, cx + 2);
  const uint32_t f_w1 = b.ld_any(flag_plane, cx - 1), f_w2 = b.ld_any(flag_plane, cx - 2);
  const uint32_t n_e1 = e1 & ~f_e1, n_e2 = e2 & ~f_e2, n_w1 = w1 & ~f_w1, n_w2 = w2 & ~f_w2;
  b.st_if(n_e1 != 0u, flag_plane, cx + 1, f_e1 | n_e1);
  b.st_if(n_e2 != 0u, flag_plane, cx + 2, f_e2 | n_e2);
  b.st_if(n_w1 != 0u, flag_plane, cx - 1, f_w1 | n_w1);
  b.st_if(n_w2 != 0u, flag_plane, cx - 2, f_w2 | n_w2);
  fresh[0] = n_e1;
  fresh[1] = n_e2;
  fresh[2] = n_w1;
  fresh[3] = n_w2;
}

template <class B, class Stack>
TW_HD void flood_visit_entry(B& b, int flag_plane, Stack& stk, uint32_t e) {
  const int cx = static_cast<int>(e >> 24);
  uint32_t fresh[4];
  flood_flag_neighbours(b, flag_plane, cx, e & 0x00FFFFFFu, fresh);
  const bool found[4] = {fresh[0] != 0u, fresh[1] != 0u, fresh[2] != 0u, fresh[3] != 0u};
  const uint32_t entries[4] = {flood_entry(cx + 1, fresh[0]), flood_entry(cx + 2, fresh[1]),
                               flood_entry(cx - 1, fresh[2]), flood_entry(cx - 2, fresh[3])};
  stk.push4_if(found, entries);
}

// A flood whose work list is a SET OF COLUMNS (the fused playout kernel): bit c of `todo` = column c holds
// cells that got the flag and may not have been expanded yet.  A visit takes the highest such column and
// expands ALL of the flooding colour's flagged cells in it (`own_plane`), not just the new ones: re-expanding
// a cell adds nothing unless its component still owes this flood, and then it only does that flood's work
// early.  That rests on the flags being uniform over every component of a colour except the one whose flood
// is running or owed, which holds for the flooding colour even after the game ends.  (It does not hold for the
// OPPONENT: a winning move that joins a START and an END component without a neutral link owes no flood, so its
// component keeps mixed flags; expanding all flagged cells of the column regardless of colour would spread them.)
// A flood starts with todo = the bit of the new peg's column and ends when todo is 0; the work list needs
// no memory and cannot overflow.
template <class B>
TW_HD void flood_visit_columns(B& b, int own_plane, int flag_plane, uint32_t& todo) {
  const int cx = tw_msb(todo);
  todo ^= 1u << cx;  // a visit flags cells of other columns only
  uint32_t fresh[4];
  flood_flag_neighbours(b, flag_plane, cx, b.ld(flag_plane, cx) & b.ld_pegs(own_plane, cx), fresh);
  // bit j of `m` = column cx + j - 2 (a column off the board never gets a flag, so its bit stays clear)
  const uint32_t m = (fresh[3] != 0u ? 1u : 0u) | (fresh[2] != 0u ? 2u : 0u) | (fresh[0] != 0u ? 8u : 0u) |
                     (fresh[1] != 0u ? 16u : 0u);
  todo |= (m << cx) >> 2;
}

// ... of the entry on top of the stack
template <class B, class Stack>
TW_HD void flood_visit(B& b, int flag_plane, Stack& stk) {
  const uint32_t e = stk.top();
  stk.pop();
  flood_visit_entry(b, flag_plane, stk, e);
}

// If the stack overflowed, the dropped cells are recovered by closing the
// flagged set of this colour under the link relation (flags are uniform per
// connected component while a game is open, so this only grows the component
// being flooded).  Rare; exercised by the tests with a 2-entry stack.
template <class B>
TW_HD_NOINLINE void flood_closure(B& b, int own_plane, int flag_plane) {
  bool changed = true;
  while (changed) {
    changed = false;
    for (int cx = 0; cx < b.n(); ++cx) {
      uint32_t w = b.ld(flag_plane, cx) & b.ld_pegs(own_plane, cx);
      while (w) {
        const int cy = tw_ctz(w);
        w &= w - 1u;
        uint32_t lm = links_of(b, cx, cy);
        while (lm) {
          const int d = tw_ctz(lm);
          lm &= lm - 1u;
          const int tx = cx + dir_dx(d), ty = cy + dir_dy(d);
          const uint32_t f = b.ld(flag_plane, tx);
          if (!((f >> ty) & 1u)) {
            b.st(flag_plane, tx, f | (1u << ty));
            changed = true;
          }
        }
      }
    }
  }
}

// The whole flood at once (apply kernel, host tests).
template <int kStack, class B>
TW_HD_NOINLINE void flood_flag(B& b, int own_plane, int flag_plane, int x, int y) {
  LocalStack<kStack> stk;
  stk.push(flood_entry(x, 1u << y));
  while (!stk.empty()) flood_visit(b, flag_plane, stk);
  if (stk.overflow) flood_closure(b, own_plane, flag_plane);
}

enum : uint32_t { kFloodStart = 1u, kFloodEnd = 2u };

// A move is evaluated in three pieces so that the fused playout kernel can
// overlap the middle one with the selection of the following move:
//   begin_move   swap handling, the peg itself, the counters, and the mask of
//                own-colour pegs a knight's move away (the link candidates)
//   link_move    SetPegAndLinks' link part (twixtboard.cc:510-556): crossing
//                tests, links / blocked flags, inherited border flags
//   finish_move  move counter, first-move bookkeeping, result (192-207)
struct Placement {
  int x, y;        // where the peg went (differs from the action's cell after a swap)
  int player;
  // own-colour pegs a knight's move away, as row masks of the columns x-2, x-1, x+1, x+2
  // (index = dx + 2; entry 2 unused): the link candidates
  uint32_t cand[5];
  uint32_t action; // the action as played
};

// The swap (twixtboard.cc:465-475): blue answers red's first move with the same action.  The red peg is
// taken back (UndoFirstMove, 450-455) and (x,y) becomes the cell turned by 90 degrees, where the blue peg
// goes (471-473).
TW_HD bool is_swap(const Header& h, uint32_t action) { return h.ply == 1u && action == h.move_one; }

template <class B>
TW_HD void swap_first_move(B& b, Header& h, int& x, int& y) {
  const int n = b.n();
  b.st_pegs(P_RED, x, b.ld_pegs(P_RED, x) & ~(1u << y));
  b.note_peg(x, y, -1);
  b.st(P_START, x, b.ld(P_START, x) & ~(1u << y));
  b.st(P_END, x, b.ld(P_END, x) & ~(1u << y));
  h.cnt[kRed] += (x >= 1 && x <= n - 2) ? 1 : 0;
  h.cnt[kBlue] += (y >= 1 && y <= n - 2) ? 1 : 0;
  h.swapped = 1u;
  const int rx = y, ry = n - 1 - x;
  x = rx;
  y = ry;
}

// kSwapDone: the caller has already run swap_first_move for a swapping action (the fused playout kernel
// does it in its rare-events block, so that the per-move code has no branch for it).
// kPreloaded: `own_word` is the mover's peg word of column x as it stands (the fused playout kernel has it in a
// register from choosing the cell, which saves a shared-memory round trip at the head of the move).
template <bool kSwapDone = false, bool kPreloaded = false, class B>
TW_HD Placement begin_move(B& b, Header& h, int x, int y, uint32_t own_word = 0u) {
  const int n = b.n();
  Placement p;
  p.player = static_cast<int>(h.ply & 1u);
  p.action = static_cast<uint32_t>(x * n + y);  // only read for the first move of a game
  if (!kSwapDone && is_swap(h, p.action)) swap_first_move(b, h, x, y);
  p.x = x;
  p.y = y;
  const int own = p.player == kRed ? P_RED : P_BLUE;
  b.st_pegs(own, x, (kPreloaded ? own_word : b.ld_pegs(own, x)) | (1u << y));
  b.note_peg(x, y, +1);
  h.cnt[kRed] -= (x >= 1 && x <= n - 2) ? 1 : 0;
  h.cnt[kBlue] -= (y >= 1 && y <= n - 2) ? 1 : 0;
  // own-colour pegs a knight's move away: rows y+-2 of the columns x+-1, rows y+-1 of the columns x+-2
  const uint32_t bit = 1u << y;
  const uint32_t rows2 = (bit << 2) | (bit >> 2), rows1 = (bit << 1) | (bit >> 1);
  p.cand[0] = b.ld_pegs_guard(own, x - 2) & rows1;
  p.cand[1] = b.ld_pegs_guard(own, x - 1) & rows2;
  p.cand[2] = 0u;
  p.cand[3] = b.ld_pegs_guard(own, x + 1) & rows2;
  p.cand[4] = b.ld_pegs_guard(own, x + 2) & rows1;
  return p;
}

// Returns true iff the new peg is now linked to both of its owner's border
// lines (the win test of UpdateResult, twixtboard.cc:194-199); `pending`
// receives kFloodStart / kFloodEnd for the floods the caller still has to run
// from the peg (twixtboard.cc:558-570).  Straight-line code: the eight
// directions are handled direction-major with compile-time offsets and crossing
// masks, all inputs fetched up front by independent loads; kAlways = true drops
// even the `any candidate?` branch so the whole function is one basic block.
template <bool kAlways, class B>
TW_HD bool link_move(B& b, const Placement& p, uint32_t& pending) {
  const int n = b.n();
  const int x = p.x, y = p.y;
  const uint32_t bit = 1u << y;
  // border flags the cell has by position (twixtboard.cc:223-231); a peg can
  // only stand on its owner's border lines
  bool to_start = p.player == kRed ? (y == 0) : (x == 0);
  bool to_end = p.player == kRed ? (y == n - 1) : (x == n - 1);
  bool neutral = false, new_links = false;
  if (kAlways || (p.cand[0] | p.cand[1] | p.cand[3] | p.cand[4])) {
    // everything the eight directions may read, fetched with independent loads
    LinkWindow lw, ly;
    uint32_t fs[5], fe[5];  // border flags of columns x-2 .. x+2
    uint32_t blk[3] = {0u, 0u, 0u};  // new blocked-east bits of columns x, x-1, x-2
    const uint32_t factor = align_factor(y);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int c = 0; c < 5; ++c) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
      for (int pl = 0; pl < 4; ++pl) {
        lw.w[pl][c] = b.ld_link(P_LINK0 + pl, x - 3 + c);
        ly.w[pl][c] = align_word(lw.w[pl][c], factor);  // the new peg's row at a fixed bit
      }
      fs[c] = b.ld_any(P_START, x - 2 + c);  // only read under made[c], which is empty off the board
      fe[c] = b.ld_any(P_END, x - 2 + c);
    }
    // crossed[c]: cells of column x-2+c the link to which would be crossed, as row masks
    uint32_t crossed[5] = {0u, 0u, 0u, 0u, 0u};
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int d = 0; d < 8; ++d) {
      const int dx = dir_dx(d), dy = dir_dy(d);
      const uint32_t tbit = dy > 0 ? (bit << dy) : (bit >> (-dy));  // the target cell's row
      crossed[dx + 2] |= crossing_blocked(ly, d) ? tbit : 0u;
    }
    // made[c] / blocked candidates per column, column-parallel
    uint32_t made[5];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int c = 0; c < 5; ++c) made[c] = p.cand[c] & ~crossed[c];
    // SetBlockedNeighbor on both ends (twixtboard.cc:550-551); only the bit pointing east is ever read
    // (twixtcell.h:82-84) and it always lands on the WEST endpoint of the refused link: the new peg
    // itself for the four east directions, the target for the west ones (columns x-1, x-2)
    blk[0] = ((p.cand[3] & crossed[3]) | (p.cand[4] & crossed[4])) ? bit : 0u;
    blk[1] = p.cand[1] & crossed[1];
    blk[2] = p.cand[0] & crossed[0];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int d = 0; d < 8; ++d) {
      const int dx = dir_dx(d), dy = dir_dy(d);
      const uint32_t tbit = dy > 0 ? (bit << dy) : (bit >> (-dy));
      // the link named by its west endpoint (column x+ow, row mask wbit) and east direction de; each
      // direction owns a distinct (plane, column) word, and links made earlier in this move never cross
      // later ones (they share the new peg)
      const int ow = d < 4 ? 0 : dx, de = d & 3;
      const uint32_t wbit = d < 4 ? bit : tbit;
      b.st_if((made[dx + 2] & tbit) != 0u, P_LINK0 + de, x + ow, lw.w[de][ow + 3] | wbit);
    }
    // what the new links reach, column-parallel: a start-flagged peg gives the start flag, otherwise an
    // end-flagged one the end flag, otherwise the link is neutral (twixtboard.cc:538-546)
    uint32_t any = 0u, hit_s = 0u, hit_e = 0u, hit_n = 0u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int c = 0; c < 5; ++c) {
      if (c == 2) continue;
      const uint32_t rest = made[c] & ~fs[c];
      any |= made[c];
      hit_s |= made[c] & fs[c];
      hit_e |= rest & fe[c];
      hit_n |= rest & ~fe[c];
    }
    new_links = any != 0u;
    to_start |= hit_s != 0u;
    to_end |= hit_e != 0u;
    neutral = hit_n != 0u;
    b.or_blocked3(x, blk);
    // the new peg's own flag words are fs[2] / fe[2]
    b.st_if(to_start, P_START, x, fs[2] | bit);
    b.st_if(to_end, P_END, x, fe[2] | bit);
  } else {
    b.st_if(to_start, P_START, x, b.ld(P_START, x) | bit);
    b.st_if(to_end, P_END, x, b.ld(P_END, x) | bit);
  }
  pending = (new_links && neutral) ? ((to_start ? kFloodStart : 0u) | (to_end ? kFloodEnd : 0u)) : 0u;
  return to_start && to_end;
}

TW_HD void finish_move(Header& h, const Placement& p, bool win) {
  if (h.ply == 0u) h.move_one = p.action;
  h.ply += 1u;
  if (win) h.result = p.player == kRed ? kRedWin : kBlueWin;   // twixtboard.cc:194-199
  else if ((p.player == kRed ? h.cnt[kBlue] : h.cnt[kRed]) == 0) h.result = kDraw;  // 203-206
}

// Board::ApplyAction (twixtboard.cc:457-499) for an action known to be legal,
// given as its cell (x,y) (action == x*n+y), up to but excluding the border-
// flag floods: on return (x,y) is the cell the peg went to (it differs from the
// action's cell after a swap) and `pending` names the floods still to run from
// it.  The result does not depend on them (the win test reads the new peg's
// own flags), so the header is final.
template <class B>
TW_HD void apply_begin(B& b, Header& h, int& x, int& y, uint32_t& pending) {
  const Placement p = begin_move(b, h, x, y);
  const bool win = link_move<false>(b, p, pending);
  finish_move(h, p, win);
  x = p.x;
  y = p.y;
}

// The complete move (apply kernel, host tests).
template <int kStack, class B>
TW_HD void apply_legal_cell(B& b, Header& h, int x, int y) {
  uint32_t pending;
  apply_begin(b, h, x, y, pending);
  if (pending) {
    const int own = ((h.ply - 1u) & 1u) == kRed ? P_RED : P_BLUE;
    if (pending & kFloodStart) flood_flag<kStack>(b, own, P_START, x, y);
    if (pending & kFloodEnd) flood_flag<kStack>(b, own, P_END, x, y);
  }
}

// Position of the k-th (0-based) set bit of w; k < popc(w).
TW_HD int select_bit(uint32_t w, int k) {
  int pos = 0, c;
  c = tw_popc(w & 0xFFFFu);
  if (k >= c) { k -= c; pos += 16; w >>= 16; }
  c = tw_popc(w & 0xFFu);
  if (k >= c) { k -= c; pos += 8; w >>= 8; }
  c = tw_popc(w & 0xFu);
  if (k >= c) { k -= c; pos += 4; w >>= 4; }
  c = tw_popc(w & 0x3u);
  if (k >= c) { k -= c; pos += 2; w >>= 2; }
  c = static_cast<int>(w & 1u);
  if (k >= c) pos += 1;
  return pos;
}

// select_bit with a table for the last step (fused playout): the byte holding the k-th set bit is found with two
// popcounts, the bit inside it by one look-up in a 2 KB table lut[rank][byte] (rank 0..7) -- 18 instructions
// instead of the 35 of the five-level search.  The accessor provides select_lut() (shared memory in the kernel).
TW_HD void fill_select_lut(uint8_t* lut, int entry) {  // entry = rank * 256 + byte
  const uint32_t byte = static_cast<uint32_t>(entry) & 255u;
  const int rank = entry >> 8;
  lut[entry] = static_cast<uint8_t>(rank < tw_popc(byte) ? select_bit(byte, rank) : 0);
}
TW_HD int select_bit_lut(const uint8_t* lut, uint32_t w, int k) {  // w < 2^24, k < popc(w)
  const int c0 = tw_popc(w & 0xFFu), c01 = tw_popc(w & 0xFFFFu);
  const bool ge0 = k >= c0, ge1 = k >= c01;
  const int byte_index = (ge0 ? 1 : 0) + (ge1 ? 1 : 0);
  const int before = ge1 ? c01 : (ge0 ? c0 : 0);
  const uint32_t byte = (w >> (8 * byte_index)) & 0xFFu;
  return 8 * byte_index + lut[(((k - before) & 7) << 8) | static_cast<int>(byte)];  // (& 7: an unused speculative rank stays in the table)
}

// ---- per-column count cache (fused playout only) ---------------------------
// Scanning 24 column words per move to find the k-th legal cell is the largest
// fixed cost of a playout step.  An accessor with kCountCache keeps, next to the
// planes, one byte per column: bits 0-4 = pegs in the column, bits 5-6 = pegs of
// the column on the two border rows (0 and n-1).  From these the mover's legal
// count of every column follows without touching the planes
//   red : n - pegs              (columns 1..n-2; twixtboard.cc:266-273)
//   blue: (n-2) - pegs + border (rows 1..n-2 of every column)
//   ply 1: n-2 for every column (blue's list is still the initial one)
// and four columns are handled per 32-bit word (bytewise arithmetic, byte prefix
// sums by one multiply).  The accessor provides cache_ld(i) / cache_st(i, v).
TW_HD uint32_t bytes4(uint32_t v) { return v * 0x01010101u; }

// 0xFF in byte j of word i iff column 4i+j is in [lo, hi]
TW_HD uint32_t column_byte_mask(int i, int lo, int hi) {
  uint32_t m = 0;
  for (int j = 0; j < 4; ++j) {
    const int x = 4 * i + j;
    if (x >= lo && x <= hi) m |= 0xFFu << (8 * j);
  }
  return m;
}

// per-byte (a > b), 0xFF / 0x00, all bytes < 0x80
TW_HD uint32_t bytes_gt(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __vcmpgtu4(a, b);
#else
  uint32_t r = 0;
  for (int j = 0; j < 4; ++j)
    if (((a >> (8 * j)) & 0xFFu) > ((b >> (8 * j)) & 0xFFu)) r |= 0xFFu << (8 * j);
  return r;
#endif
}

template <class B>
TW_HD void count_cache_build(B& b) {
  const int n = b.n();
  const uint32_t border = 1u | (1u << (n - 1));
  for (int i = 0; i < (n + 3) / 4; ++i) {
    uint32_t w = 0;
    for (int j = 0; j < 4; ++j) {
      const int x = 4 * i + j;
      if (x < n) {
        const uint32_t occ = b.ld_pegs(P_RED, x) | b.ld_pegs(P_BLUE, x);
        w |= static_cast<uint32_t>(tw_popc(occ) | (tw_popc(occ & border) << 5)) << (8 * j);
      }
    }
    b.cache_st(i, w);
  }
}

// Legal cells per column of the player to move, four columns per word, from cache word i.  What depends on
// the position's mode (ply 1 / red to move / blue to move) is folded into three constants chosen once per
// selection, so each word costs five instructions:
//   count4 = (base4 - (w & pegm) + ((w >> 5) & brdm)) & columns_i
//   ply 1: base4 = n-2, pegm = brdm = 0     (the full initial list, every column)
//   red  : base4 = n,   pegm = pegs, brdm = 0   (columns 1..n-2)
//   blue : base4 = n-2, pegm = pegs, brdm = border pegs (every column)
struct CountMode {
  uint32_t base4, pegm, brdm;
  bool red;
};
TW_HD CountMode count_mode(const Header& h, int n) {
  const bool first = h.ply == 1u;
  const bool red = !first && (h.ply & 1u) == kRed;
  CountMode m;
  m.base4 = bytes4(static_cast<uint32_t>(red ? n : n - 2));
  m.pegm = first ? 0u : 0x1F1F1F1Fu;
  m.brdm = (first || red) ? 0u : 0x03030303u;
  m.red = red;
  return m;
}
TW_HD uint32_t count_cache_legal4(uint32_t w, const CountMode& m, int n, int i) {
  const uint32_t inner = column_byte_mask(i, 1, n - 2), every = column_byte_mask(i, 0, n - 1);
  const uint32_t columns = inner == every ? every : (m.red ? inner : every);  // differs in the two edge words only
  return (m.base4 - (w & m.pegm) + ((w >> 5) & m.brdm)) & columns;
}

template <class B>
TW_HD void select_legal_cached(const B& b, const Header& h, int k, int& out_x, int& out_y, uint32_t* out_pegs = nullptr) {
  const int n = b.n();
  constexpr int kMaxWords = 6;  // ceil(24 / 4)
  const int words = (n + 3) / 4;
  // all cache words first (independent loads), then the arithmetic
  uint32_t cw[kMaxWords];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int i = 0; i < kMaxWords; ++i) cw[i] = i < words ? b.cache_ld(i) : 0u;
  const CountMode mode = count_mode(h, n);
  uint32_t sp = 0;  // byte prefix sums of the selected word
  int si = 0, sk = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int i = 0; i < kMaxWords; ++i) {
    if (i < words) {
      const uint32_t p4 = count_cache_legal4(cw[i], mode, n, i) * 0x01010101u;  // inclusive byte prefix sums
      if (k >= 0) { sp = p4; si = i; sk = k; }
      k -= static_cast<int>(p4 >> 24);
    }
  }
  // first byte whose inclusive prefix exceeds sk.  The bytes of sp are prefix sums, i.e. non-decreasing, so that
  // byte's index is the NUMBER of bytes not above sk: three independent compares (the fourth byte is above sk for
  // every valid k) instead of a bytewise compare emulated in six dependent instructions plus a find-first-set --
  // this is the tail of the playout kernel's loop-carried selection chain.  `before` = the prefix of the byte
  // in front of it.  (With no legal cell at all -- a speculative selection that is never used -- j = 3 and the
  // clamp below keeps the loads on the board.)
  const int p0 = static_cast<int>(sp & 0xFFu), p1 = static_cast<int>((sp >> 8) & 0xFFu), p2 = static_cast<int>((sp >> 16) & 0xFFu);
  const bool le0 = p0 <= sk, le1 = p1 <= sk, le2 = p2 <= sk;
  const int j = (le0 ? 1 : 0) + (le1 ? 1 : 0) + (le2 ? 1 : 0);
  const int before = le2 ? p2 : (le1 ? p1 : (le0 ? p0 : 0));
  const int x = (4 * si + j) < n ? (4 * si + j) : (n - 1);
  out_x = x;
  if constexpr (B::kSelectLut) {
    // (a speculative selection with no legal cell left may land on an edge column: the masks below keep the
    // look-up inside the table, and its result is never used)
    const uint32_t red = b.ld_pegs(P_RED, x), blue = b.ld_pegs(P_BLUE, x);
    if (out_pegs != nullptr) {  // the chosen column's peg words, for begin_move<.., kPreloaded>
      out_pegs[0] = red;
      out_pegs[1] = blue;
    }
    const uint32_t play = (h.ply & 1u) == kRed ? full_rows(n) : inner_rows(n);  // (legal_word_selected, spelled out)
    const uint32_t w = (h.ply == 1u ? play : (play & ~(red | blue))) & 0xFFFFFFu;
    out_y = select_bit_lut(b.select_lut(), w, sk - before);
  } else {
    out_y = select_bit(legal_word(b, h, x), sk - before);
  }
}

// The k-th action (0-based) of the ascending legal list, as a cell; k <
// legal_count.  Ascending action order is column-major (action = x*n+y,
// twixtboard.cc:603-605), i.e. the order of the column words.
template <class B>
TW_HD void select_legal(const B& b, const Header& h, int k, int& out_x, int& out_y, uint32_t* out_pegs = nullptr) {
  if constexpr (B::kCountCache) {
    select_legal_cached(b, h, k, out_x, out_y, out_pegs);
  } else {
    int sx = 0, sk = 0;
    uint32_t sw = 0;
    for (int x = 0; x < b.n(); ++x) {
      uint32_t w = legal_word(b, h, x);
      if (k >= 0) { sx = x; sw = w; sk = k; }
      k -= tw_popc(w);
    }
    out_x = sx;
    out_y = select_bit(sw, sk);
  }
}

// Column word of "peg has at least one link" (Cell::HasLinks, twixtcell.h:78).
template <class B>
TW_HD uint32_t haslink_word(const B& b, int x) {
  uint32_t m = b.ld(P_LINK0 + 0, x) | b.ld(P_LINK0 + 1, x) | b.ld(P_LINK0 + 2, x) | b.ld(P_LINK0 + 3, x);
  m |= b.ld_guard(P_LINK0 + 0, x - 1) << 2;
  m |= b.ld_guard(P_LINK0 + 1, x - 2) << 1;
  m |= b.ld_guard(P_LINK0 + 2, x - 2) >> 1;
  m |= b.ld_guard(P_LINK0 + 3, x - 1) >> 2;
  return m;
}

// Column word (over y) of observation plane `plane` (0..11) in BOARD
// coordinates: which cells (x, .) put a 1.0 into that plane
// (SetPegAndLinksOnTensor, twixt.cc:76-99).
template <class B>
TW_HD uint32_t obs_plane_word(const B& b, int plane, int x) {
  const int own = plane < 6 ? P_RED : P_BLUE;
  const int k = plane < 6 ? plane : plane - 6;
  const uint32_t pegs = b.ld_pegs(own, x);
  if (k == 0) return pegs & ~haslink_word(b, x);
  if (k == 5) return pegs & b.ld(P_BLOCKED, x);
  return pegs & b.ld(P_LINK0 + (k - 1), x);
}

// Board cell feeding tensor element (plane, r, c) (GetTensorPosition,
// twixtboard.cc:590-597, inverted): red planes are the board seen from above
// without red's... opponent's end columns, blue planes are turned by 90 degrees.
TW_HD void obs_cell(int n, int plane, int r, int c, int& x, int& y) {
  if (plane < 6) { x = c + 1; y = n - 1 - r; }
  else { x = n - 1 - r; y = n - 2 - c; }
}

}  // namespace twixt
