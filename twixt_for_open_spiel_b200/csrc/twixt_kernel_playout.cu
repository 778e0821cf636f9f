// twixt_kernel_playout.cu -- K5, the fused random-playout kernel.
//
// One THREAD per env.  Each lane copies the bit-planes of its env from HBM into
// shared memory, transposed so that word w of lane l sits at smem[w*32 + l]:
// whatever word each lane indexes, lane l always hits bank l, so every access
// of the scalar rules in twixt_engine.cuh is conflict-free.  The whole game is
// then played out of shared memory -- select a uniformly random legal action
// (Philox4x32-10, one block per four moves), apply it (peg, links, crossing
// test, border flags, result) -- and the final planes are written back once.
// HBM sees 2 x record bytes per GAME, not per move; the limiter is issue slots
// and shared-memory latency, which is why the thread-per-env mapping is used:
// it spends ~1/10 of the warp-instructions per move of a warp-per-env mapping
// because nothing is computed redundantly across lanes (DESIGN.md, "Mapping
// one game onto the machine").
//
// Divergence control (profiles/r1_playout_v1_*: 9.5 of 32 lanes active):
//  * the border-flag flood (ExploreLocalGraph) is cut into single visits that
//    are interleaved with the other lanes' moves: every loop iteration runs
//    one MOVE for the lanes without flood work and one flood VISIT for the
//    lanes with it, instead of 31 lanes idling through one lane's whole flood;
//    its work list is one register, the set of columns still to expand
//    (flood_visit_columns);
//  * candidate links are handled direction-major and branch-free (link_move),
//    a flood visit handles a whole column at once;
//  * lanes are PERSISTENT: games end at different plies (250..573 at n=24), so
//    a lane whose game is over writes its env back and takes the next env of
//    the range from a ticket counter instead of idling until the slowest game
//    of its warp ends; the new env arrives by cp.async (LDGSTS) while the rest
//    of the warp keeps playing.
// Control structure (profiles/r1_playout_v15_* -> v18_*): with two warps per
// scheduler every reconvergence point shows up as a stall, so an iteration has
// exactly three data-dependent branch regions -- RARE (finish a load, retire
// an env and take the next, first half of a swap), MOVE, FLOOD -- plus the
// warp-uniform Philox refresh / loop-exit vote every fourth iteration.
// Shared memory per env: the planes BLUE, RED, links x4, START, END (this
// order puts an always-zero word in front of every link plane, so the link
// window of a move is loaded without bounds tests) + 4 pad words (8n + 4 words,
// 784 B at n = 24: nine warps fit on an SM); the
// per-column count cache that replaces the 24-word legal scan by 6 bytewise
// words (twixt_engine.cuh, count_cache_*) lives in registers.  The "blocked
// neighbour" plane is write-only for the rules, so it stays in HBM and is
// OR-ed in place (RED.OR, fire-and-forget).
//
// Reference loop reproduced: upstream example.cc / RandomRolloutEvaluator
// (LegalActions -> uniform pick -> ApplyAction until IsTerminal), with the
// per-move semantics of twixtboard.cc:457-499.
#include <cuda_pipeline.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <cstdlib>

#include "twixt_b200.h"
#include "twixt_engine.cuh"
#include "twixt_kernels.cuh"
#include "twixt_philox.cuh"

namespace twixt {

namespace {

#ifndef TW_PLAYOUT_THREADS
#define TW_PLAYOUT_THREADS 128
#endif
#ifndef TW_PLAYOUT_MIN_BLOCKS
#define TW_PLAYOUT_MIN_BLOCKS 1
#endif
constexpr int kPlayoutThreads = TW_PLAYOUT_THREADS;  // 4 warps per block (the default; see playout_threads)
constexpr int kSmemPlanes = 8;        // P_RED .. P_END
// Words behind the END plane.  The rules' unguarded flag loads (ld_any in link_move and the flood visit) read
// END at columns n and n+1, which land here instead of leaving the lane's column; and while an env is being
// loaded its header is parked here (the loads' values are ignored, so whatever they find is harmless).
constexpr int kPadWords = 4;
constexpr int kCacheWords = 6;        // per-column count cache, four columns per word
constexpr int kSelectLutBytes = 8 * 256;  // select_bit_lut: [rank 0..7][byte]
constexpr unsigned kFullMask = 0xFFFFFFFFu;

// words of shared memory per env: the planes and the pad words; the run-time-size form (never instantiated,
// see PlayoutRef) would keep its count cache there too
__host__ __device__ constexpr int playout_words(int n, bool cache_in_smem = false) {
  return kSmemPlanes * n + kPadWords + (cache_in_smem ? kCacheWords : 0);
}

// -DTW_PLAYOUT_BOUNDS_CHECK=1 builds the INSTRUMENTED variant used by tests/ (never the product build): every
// shared-memory access of the rules is tested against the lane's own column,
// [0, playout_words) words, and every blocked-plane reduction against [0, n); a violation is counted in
// DeviceStats::bounds_violations (twixt_stats.debug_violations) and the access is redirected to word 0 /
// column 0, so a broken invariant shows up as a number instead of a fault.  The unguarded link-window and
// flag loads are ALLOWED to leave the board (they land in this env's neighbouring planes or pad words,
// see ld_link / ld_any below) but never the lane's column: that is what this variant proves.
#ifndef TW_PLAYOUT_BOUNDS_CHECK
#define TW_PLAYOUT_BOUNDS_CHECK 0
#endif
#ifndef TW_FLOOD_OVERLAP
#define TW_FLOOD_OVERLAP 1
#endif
// -DTW_PLAYOUT_MAX_BLOCKS=b (b > 0) caps the persistent grid at b blocks: a TEST variant (never the product
// build) in which every lane plays many envs in a row through the ticket counter, so the hand-over from one
// game to the next is exercised ten or more times per lane instead of once or twice.
#ifndef TW_PLAYOUT_MAX_BLOCKS
#define TW_PLAYOUT_MAX_BLOCKS 0
#endif

// The env's planes in shared memory (stride 32 words) + its blocked plane in HBM.
template <int NT>
struct PlayoutRef {
  uint32_t* p;     // smem, this lane's column
  uint32_t* gblk;  // global: the record's P_BLOCKED words
#if TW_PLAYOUT_BOUNDS_CHECK
  unsigned long long* viol;
  __device__ __forceinline__ int chk(int word) const {
    if (word < 0 || word >= playout_words(n(), NT == 0)) {
      atomicAdd(viol, 1ull);
      return 0;
    }
    return word;
  }
  __device__ __forceinline__ int chk_col(int col) const {
    if (col < 0 || col >= n()) {
      atomicAdd(viol, 1ull);
      return 0;
    }
    return col;
  }
#else
  __device__ __forceinline__ int chk(int word) const { return word; }
  __device__ __forceinline__ int chk_col(int col) const { return col; }
#endif
  // NT is the board size (every size 5..24 is instantiated, see the end of the file).  The run-time-size
  // form (NT == 0, n_rt, count cache in shared memory) is no longer instantiated; it is kept because taking
  // it out changed ptxas' schedule of the n = 24 kernel for the worse (18.4 -> 18.8 ms, measured twice).
  int n_rt;
  __device__ __forceinline__ int n() const { return NT > 0 ? NT : n_rt; }
  // Shared-memory order of the planes: BLUE, RED, the four link planes, START, END (the record has RED
  // first).  With it the word in front of every link plane is always zero -- red never stands in column
  // n-1 (blue's end line), and a link plane holds links at their WEST endpoint, so its column n-1 is
  // empty -- which is what ld_link needs: the rules' link-window loads carry no bounds test at all.  Words
  // read further off the board belong to this env's neighbouring planes or its pad words.
  __device__ __forceinline__ uint32_t ld(int plane, int col) const { return p[chk(plane * n() + col) * 32]; }
  __device__ __forceinline__ void st(int plane, int col, uint32_t v) { p[chk(plane * n() + col) * 32] = v; }
  __device__ __forceinline__ uint32_t ld_link(int plane, int col) const { return ld(plane, col); }
  __device__ __forceinline__ uint32_t ld_any(int plane, int col) const { return ld(plane, col); }
  // record word (after the header) -> shared-memory word
  __device__ __forceinline__ int smem_word(int w) const { return w < n() ? w + n() : (w < 2 * n() ? w - n() : w); }
  // conditional plane store as ONE predicated st.shared: the compiler turns `if (c) st(...)` into a
  // BSSY/BRA/BSYNC region (ten of them per move showed up as branch_resolving stalls), and redirecting
  // the store of the "false" lanes to a spare word measured slower than that
  __device__ __forceinline__ void st_if(bool c, int plane, int col, uint32_t v) {
    const int word = c ? chk(plane * n() + col) : plane * n() + col;  // only a store that happens is an access
    const uint32_t addr = static_cast<uint32_t>(__cvta_generic_to_shared(p + word * 32));
    asm volatile(
        "{\n\t.reg .pred pp;\n\tsetp.ne.u32 pp, %0, 0;\n\t@pp st.shared.u32 [%1], %2;\n\t}"
        :: "r"(static_cast<uint32_t>(c)), "r"(addr), "r"(v) : "memory");
  }
  __device__ __forceinline__ uint32_t ld_guard(int plane, int col) const {
    return (static_cast<unsigned>(col) < static_cast<unsigned>(n())) ? ld(plane, col) : 0u;
  }
  __device__ __forceinline__ uint32_t ld_pegs(int plane, int col) const { return ld(plane ^ 1, col); }
  __device__ __forceinline__ void st_pegs(int plane, int col, uint32_t v) { st(plane ^ 1, col, v); }
  __device__ __forceinline__ uint32_t ld_pegs_guard(int plane, int col) const { return ld_guard(plane ^ 1, col); }
  // fire-and-forget reduction (RED.OR): no load to wait for; only this thread touches the word
  __device__ __forceinline__ void or_blocked(int col, uint32_t bits) { atomicOr(gblk + chk_col(col), bits); }
  // Three UNCONDITIONAL reductions per move: OR-ing zero bits is harmless (and a column left of the board
  // only ever gets zero bits: its address is clamped).  ptxas cannot predicate a RED -- every conditional
  // one becomes its own branch region (three of them cost 9 %), and even one branch around all three
  // (taken by half of the moves) was 2.5 % slower than always issuing them.
  __device__ __forceinline__ void or_blocked3(int x, const uint32_t blk[3]) {
    atomicOr(gblk + chk_col(x), blk[0]);
    atomicOr(gblk + chk_col(max(x - 1, 0)), blk[1]);
    atomicOr(gblk + chk_col(max(x - 2, 0)), blk[2]);
  }
  // per-column count cache (twixt_engine.cuh, count_cache_*).  With a compile-time board size every index
  // into it is static after unrolling, so the six words live in REGISTERS (no load before a selection, no
  // store->load round trip after a move); the run-time-size instantiation keeps them in shared memory
  // after the planes and the pad words.
  static constexpr bool kCountCache = true;
  static constexpr bool kSelectLut = true;
  const uint8_t* lut;  // shared memory: select_bit_lut's table, filled once per block
  __device__ __forceinline__ const uint8_t* select_lut() const { return lut; }
  static constexpr bool kCacheInRegs = NT > 0;
  uint32_t cw[kCacheWords];
  __device__ __forceinline__ uint32_t* cache_word(int i) const { return p + (kSmemPlanes * n() + kPadWords + i) * 32; }
  __device__ __forceinline__ uint32_t cache_ld(int i) const { return kCacheInRegs ? cw[i] : *cache_word(i); }
  __device__ __forceinline__ void cache_st(int i, uint32_t v) {
    if (kCacheInRegs) cw[i] = v;
    else *cache_word(i) = v;
  }
  __device__ __forceinline__ void note_peg(int x, int y, int delta) {
    const uint32_t inc = (1u | ((y == 0 || y == n() - 1) ? 32u : 0u)) << (8 * (x & 3));
    const uint32_t signed_inc = delta > 0 ? inc : 0u - inc;
    if (kCacheInRegs) {
#pragma unroll
      for (int i = 0; i < kCacheWords; ++i) cw[i] += (i == (x >> 2)) ? signed_inc : 0u;
    } else {
      uint32_t* w = cache_word(x >> 2);
      *w += signed_inc;
    }
  }
};

// Block geometry per board size.  The resident warps per SM are what this latency-bound kernel lives on
// (profiles/r2_playout_occupancy_scaling.txt), and they are capped by shared memory: blocks of 128 threads
// (with 1 KB reserved per block) leave room unused at the sizes where two of them fit but three do not.  For
// those sizes ONE block of 9 or 10 warps is used instead (10 is what 195 registers per thread allow):
// measured at n = 16, 28.8 -> 30.6 G steps/s.  With 8n + 4 words per env that gives 9 warps at n = 22..24,
// 10 at n = 18..21, 12 (three blocks of 128, 170 registers) at n = 13..17 and 16 (four blocks, 128 registers)
// at n <= 12.  ptxas fits every size into its register cap without spilling, and each of these counts was
// measured faster than the previous layout's smaller one (profiles/r3_playout_flood_columns_ab.txt).
constexpr int kBlockOverhead = 1024 + 8 * 256;  // reserved by CUDA + the select table
__host__ __device__ constexpr int playout_blocks_of_128(int nt) { return (227 * 1024) / (128 * playout_words(nt) * 4 + kBlockOverhead); }
__host__ __device__ constexpr int playout_one_block_warps(int nt) {
  return ((227 * 1024 - kBlockOverhead) / (playout_words(nt) * 4)) / 32 > 10 ? 10 : ((227 * 1024 - kBlockOverhead) / (playout_words(nt) * 4)) / 32;
}
__host__ __device__ constexpr int playout_threads(int nt) {
  return (TW_PLAYOUT_THREADS != 128 || nt == 0)           ? TW_PLAYOUT_THREADS  // (experiments: a forced block size)
         : (playout_blocks_of_128(nt) == 2 && playout_one_block_warps(nt) > 8) ? 32 * playout_one_block_warps(nt)
                                                                                : 128;
}
__host__ __device__ constexpr int playout_min_blocks(int nt) {
  return nt == 0 ? TW_PLAYOUT_MIN_BLOCKS
                 : (227 * 1024) / (playout_threads(nt) * playout_words(nt) * 4 + kBlockOverhead) > 4
                       ? 4
                       : (227 * 1024) / (playout_threads(nt) * playout_words(nt) * 4 + kBlockOverhead);
}

// kTrace: write the action trace (only parity tests ask for it; the branch is compiled out otherwise)
template <int NT, bool kTrace>
__global__ void __launch_bounds__(playout_threads(NT), playout_min_blocks(NT)) playout_kernel(const PlayoutArgs a) {
  constexpr int kThreads = playout_threads(NT);
  extern __shared__ uint4 smem_raw[];
  uint32_t* smem = reinterpret_cast<uint32_t*>(smem_raw);
  const int n = NT > 0 ? NT : a.n;
  const int rw = record_words(n);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t* mine = smem + warp * (playout_words(n, NT == 0) * 32) + lane;
  const int plane_quads = (kSmemPlanes * n) / 4;  // 8n staged words = 2n 16-byte pieces (planes start 16-byte aligned)
  const uint32_t k_lo = static_cast<uint32_t>(a.seed), k_hi = static_cast<uint32_t>(a.seed >> 32);

  // ---- per-lane state of the env being played ------------------------------
  int64_t idx = -1;  // env held by this lane (index within the range), -1 = none
  uint32_t* grec = nullptr;
  Header h;
  h.ply = 0; h.result = kDraw; h.swapped = 0; h.move_one = kNoMove; h.cnt[0] = h.cnt[1] = 0;
  PlayoutRef<NT> b;
  b.p = mine;
  b.gblk = nullptr;
  b.n_rt = n;
  {
    // the 2 KB look-up table of select_bit_lut behind the env columns (the only block-wide step of the kernel)
    uint8_t* lut = reinterpret_cast<uint8_t*>(smem + kThreads * playout_words(n, NT == 0));
    for (int e = threadIdx.x; e < kSelectLutBytes; e += kThreads) fill_select_lut(lut, e);
    __syncthreads();
    b.lut = lut;
  }
#pragma unroll
  for (int i = 0; i < kCacheWords; ++i) b.cw[i] = 0u;
  uint32_t* const pad = mine + kSmemPlanes * n * 32;  // the pad words (see kPadWords)
#if TW_PLAYOUT_BOUNDS_CHECK
  b.viol = &a.stats->bounds_violations;
#endif
  uint32_t s_lo = 0, s_hi = 0;
  // Random words: block `rq` (moves 4rq..4rq+3) in ra[], block rq+1 in rb[].  Lanes of a warp are at
  // different move numbers, so blocks are produced on a warp-uniform schedule (every 4th iteration, all
  // lanes together) instead of whenever a lane runs dry, which would run the Philox rounds divergently in
  // nearly every iteration.  A lane makes at most one move per iteration, so two blocks always suffice.
  uint32_t ra[4] = {0, 0, 0, 0}, rb[4] = {0, 0, 0, 0};
  uint32_t rq = 0;
  auto word_at = [&](uint32_t index) {  // random word of move `index`, 4rq <= index < 4rq + 8
    const uint32_t rel = index - 4u * rq;
    const uint32_t wa = (rel & 2u) ? ((rel & 1u) ? ra[3] : ra[2]) : ((rel & 1u) ? ra[1] : ra[0]);
    const uint32_t wb = (rel & 2u) ? ((rel & 1u) ? rb[3] : rb[2]) : ((rel & 1u) ? rb[1] : rb[0]);
    return (rel & 4u) ? wb : wa;
  };
  // The cell of the NEXT move is chosen one move ahead: between placing a peg and evaluating its links
  // (two independent dependency chains the scheduler can interleave), see the MOVE section.
  int sx = 0, sy = 0;
  // the red / blue peg words of column sx as they stand (read while choosing the cell): begin_move takes the
  // mover's from here instead of loading it again at the head of the loop-carried select -> place chain
  uint32_t spegs[2] = {0u, 0u};
  int step = 0;
  // Border-flag floods owed: bits (2c, 2c+1) of `pend` = colour c still has to flood the START / END flag from
  // its newest peg, whose column bit is origin_r / origin_b; `todo` is the work list of the running flood (the
  // columns still to visit, flood_visit_columns) and `fcol` its colour.  A flood of
  // colour c only ever sets flag bits of c's pegs and walks c's links, and a move of the OTHER colour only
  // reads the flags of its own pegs (link_move masks them with its candidates), so the opponent moves while
  // c's flood is still running; only c's own next move has to wait for it (TW_FLOOD_OVERLAP, modelled with
  // tools/warp_sim.cc before it was built: 4 - 5 % fewer loop iterations at n = 24).
  uint32_t pend = 0, todo = 0, origin_r = 0, origin_b = 0, swapped_before = 0, fcol = 0;
  int fplane = P_START;
  bool playing = false, open_at_start = false;
  // the chosen cell is the swap (blue repeats red's first action): its first half -- taking the red peg
  // back and turning the cell -- runs in the rare-events block, so MOVE has no branch for it
  bool swap_next = false;
  int sact = 0;  // the chosen action as played (only the trace needs it: a swap turns (sx, sy))
  // ---- per-lane totals over all envs this lane plays -------------------------
  uint32_t t_plies = 0, t_games = 0, t_red = 0, t_blue = 0, t_draws = 0, t_swaps = 0, t_maxlen = 0;

  // Taking env `e` of the range is split in two so that its HBM latency overlaps the other lanes' work:
  // begin_take issues asynchronous global->shared copies (cp.async, 4 bytes each: the destination is this
  // lane's strided column) of the header (parked in the pad words) and the planes;
  // finish_take runs at the top of the next loop iteration, when the data has normally arrived.
  bool loading = false;
  bool have = false;  // this lane holds an env (idx >= 0; a flag, because the 64-bit compare sat in every iteration's top)
  auto begin_take = [&](int64_t e) {
    idx = e;
    have = true;
    grec = a.records + e * rw;
    for (int w = 0; w < kHeaderWords; ++w) __pipeline_memcpy_async(pad + w * 32, grec + w, 4);
    for (int w = 0; w < kSmemPlanes * n; ++w) __pipeline_memcpy_async(mine + b.smem_word(w) * 32, grec + kHeaderWords + w, 4);
    __pipeline_commit();
    loading = true;
    playing = false;
    pend = 0;
    todo = 0;
  };
  auto finish_take = [&]() {
    __pipeline_wait_prior(0);
    unpack_header(pad[0], pad[32], pad[64], pad[96], h);
    b.gblk = grec + kHeaderWords + P_BLOCKED * n;
    const uint64_t stream = a.stream_ids != nullptr ? a.stream_ids[idx] : a.stream_base + static_cast<uint64_t>(idx);
    s_lo = static_cast<uint32_t>(stream);
    s_hi = static_cast<uint32_t>(stream >> 32);
    step = 0;
    // Only the first block of random words is made here, where one lane runs alone: it is parked as the
    // SECOND buffered block of block number -1, so the warp-wide refresh below (at most three iterations
    // away, before word 4 is needed) shifts it into place and makes block 1 together with the other lanes'.
    rq = 0xFFFFFFFFu;
    philox4x32_10(s_lo, s_hi, 0u, 0u, k_lo, k_hi, rb);
    swapped_before = h.swapped;
    open_at_start = h.result == kOpen;
    playing = open_at_start && a.max_plies > 0;
    if (h.ply == 0u) {
      // a fresh game: no pegs to count, and red's k-th legal cell is known in closed form (every row of
      // the columns 1 .. n-2, twixtboard.cc:252-276)
#pragma unroll
      for (int i = 0; i < kCacheWords; ++i) b.cache_st(i, 0u);
      const int k = static_cast<int>(playout_index(word_at(0u), static_cast<uint32_t>(n * (n - 2))));
      sx = 1 + k / n;
      sy = k - (sx - 1) * n;
      spegs[0] = spegs[1] = 0u;  // an empty board
    } else {
      count_cache_build(b);
      if (playing)
        select_legal(b, h, static_cast<int>(playout_index(word_at(0u), static_cast<uint32_t>(legal_count(h, n)))), sx, sy, spegs);
    }
    sact = sx * n + sy;
    swap_next = playing && is_swap(h, static_cast<uint32_t>(sact));
    loading = false;
  };

  // Give the env back: final planes + header to HBM, per-env outputs, lane totals.
  auto give = [&]() {
    uint4* dst = reinterpret_cast<uint4*>(grec);
    uint4 hw;
    pack_header(h, hw.x, hw.y, hw.z, hw.w);
    dst[0] = hw;
    for (int q = 0; q < plane_quads; ++q) {
      uint4 v;
      v.x = mine[b.smem_word(4 * q + 0) * 32];
      v.y = mine[b.smem_word(4 * q + 1) * 32];
      v.z = mine[b.smem_word(4 * q + 2) * 32];
      v.w = mine[b.smem_word(4 * q + 3) * 32];
      dst[1 + q] = v;
    }
    if (a.out_returns != nullptr) {
      const float r = h.result == kRedWin ? 1.0f : (h.result == kBlueWin ? -1.0f : 0.0f);
      reinterpret_cast<float2*>(a.out_returns)[idx] = make_float2(r, r == 0.0f ? 0.0f : -r);
    }
    if (a.out_lengths != nullptr) a.out_lengths[idx] = step;
    t_plies += static_cast<uint32_t>(step);
    if (open_at_start && h.result != kOpen) {
      t_games += 1;
      t_red += h.result == kRedWin;
      t_blue += h.result == kBlueWin;
      t_draws += h.result == kDraw;
      t_maxlen = max(t_maxlen, h.ply);
    }
    t_swaps += h.swapped != swapped_before;
    idx = -1;
    have = false;
  };

  // every thread only ever touches its own column of the staging buffer: no barrier needed anywhere.
  // Tickets: the first gridDim.x*blockDim.x envs are pre-assigned, the rest are handed out by a counter.
  const int64_t preassigned = static_cast<int64_t>(gridDim.x) * kThreads;
  bool exhausted = false;
  {
    const int64_t e = blockIdx.x * static_cast<int64_t>(kThreads) + threadIdx.x;
    if (e < a.count) begin_take(e);
    else exhausted = true;
  }

  for (uint32_t it = 1;; ++it) {
    // ---- RARE (one branch region): an env whose copy was started an iteration ago is unpacked; a finished
    // env goes back to HBM and the lane starts copying the next one
    {
      const bool done = have && !loading && !playing && pend == 0u && todo == 0u;
      if (loading || done || swap_next) {
        if (loading) {
          finish_take();
        } else if (done) {
          give();
          if (!exhausted) {
            const int64_t e = preassigned + static_cast<int64_t>(atomicAdd(a.tickets, 1ull));
            if (e < a.count) begin_take(e);
            else exhausted = true;
          }
        }
        if (swap_next) {  // possibly set by finish_take just now: a game taken over at ply 1
          swap_first_move(b, h, sx, sy);  // takes the red peg back and turns (sx, sy): another column
          spegs[0] = b.ld_pegs(P_RED, sx);
          spegs[1] = b.ld_pegs(P_BLUE, sx);
          swap_next = false;
        }
      }
    }
    if ((it & 3u) == 0u) {  // warp-uniform
      // a lane only runs out of envs in the rare block above, so looking every fourth iteration is enough
      if (!__any_sync(kFullMask, have)) break;
      // every lane that has moved into its second block of random words gets the next one
      if (static_cast<uint32_t>(step) + 1u >= 4u * (rq + 1u)) {  // step+1 = next word to be consumed
        rq += 1u;
        ra[0] = rb[0]; ra[1] = rb[1]; ra[2] = rb[2]; ra[3] = rb[3];
        philox4x32_10(s_lo, s_hi, rq + 1u, 0u, k_lo, k_hi, rb);
      }
    }
    // ---- MOVE: lanes whose colour to move owes no flood make their next move -----------
#if TW_FLOOD_OVERLAP
    const uint32_t mover = h.ply & 1u;
    const bool flood_blocks = ((pend >> (2u * mover)) & 3u) != 0u || (todo != 0u && fcol == mover);
#else
    const bool flood_blocks = pend != 0u || todo != 0u;
#endif
    if (playing && !flood_blocks) {
      if (kTrace && step < a.trace_plies)
        a.out_actions[static_cast<int64_t>(step) * a.count + idx] = static_cast<uint16_t>(sact);
      const Placement pl = begin_move</*kSwapDone=*/true, /*kPreloaded=*/true>(b, h, sx, sy, (h.ply & 1u) == kRed ? spegs[0] : spegs[1]);
      // choose the following move now (speculatively: unused if this move ends the game); it only reads the
      // peg planes and the count cache, which begin_move has just brought up to date
      Header hn = h;
      hn.ply = h.ply + 1u;
      const int ln = legal_count(hn, n);
      int nx, ny;
      select_legal(b, hn, static_cast<int>(playout_index(word_at(static_cast<uint32_t>(step) + 1u), static_cast<uint32_t>(ln))), nx, ny, spegs);
      uint32_t owed;
      const bool win = link_move</*kAlways=*/true>(b, pl, owed);
      finish_move(h, pl, win);
      pend |= owed << (2 * pl.player);
      const uint32_t peg_col = 1u << pl.x;
      origin_r = pl.player == kRed ? peg_col : origin_r;
      origin_b = pl.player == kRed ? origin_b : peg_col;
      ++step;
      playing = h.result == kOpen && step < a.max_plies;
      sx = nx;
      sy = ny;
      sact = nx * n + ny;
      swap_next = playing && is_swap(h, static_cast<uint32_t>(sact));
    }
    // ---- FLOOD: one visit for the lanes that owe border-flag propagation -----
    // One branch for "start the next pending flood" and "continue the running one": a lane with no running
    // flood that owes one starts it from the new peg's column, the others visit the next column of theirs.
    if (todo != 0u || pend != 0u) {
      const bool begin = todo == 0u;
      // the next flood to start: the lowest owed one (red START, red END, blue START, blue END) -- any order
      // gives the same planes, and this one is three instructions (the "colour that moves next first" rule it
      // replaces cost a dozen with its variable shifts, for 0.1 % fewer iterations in tools/warp_sim.cc)
      const uint32_t lsb = pend & (0u - pend);
      const bool blue = (lsb & 12u) != 0u;
      fplane = begin ? ((lsb & 5u) != 0u ? P_START : P_END) : fplane;
      fcol = begin ? (blue ? 1u : 0u) : fcol;
      pend ^= begin ? lsb : 0u;
      todo = begin ? (blue ? origin_b : origin_r) : todo;
      flood_visit_columns(b, fcol == kRed ? P_RED : P_BLUE, fplane, todo);
    }
  }

  // batch statistics: warp-reduce, one atomic per warp and counter
  if (a.stats != nullptr) {
    unsigned long long plies = t_plies;
    unsigned games = t_games, red = t_red, blue = t_blue, draws = t_draws, swaps = t_swaps, maxlen = t_maxlen;
    for (int o = 16; o > 0; o >>= 1) {
      plies += __shfl_xor_sync(kFullMask, plies, o);
      games += __shfl_xor_sync(kFullMask, games, o);
      red += __shfl_xor_sync(kFullMask, red, o);
      blue += __shfl_xor_sync(kFullMask, blue, o);
      draws += __shfl_xor_sync(kFullMask, draws, o);
      swaps += __shfl_xor_sync(kFullMask, swaps, o);
      maxlen = max(maxlen, __shfl_xor_sync(kFullMask, maxlen, o));
    }
    if (lane == 0) {
      if (plies) atomicAdd(&a.stats->plies, plies);
      if (games) atomicAdd(&a.stats->games, static_cast<unsigned long long>(games));
      if (red) atomicAdd(&a.stats->red_wins, static_cast<unsigned long long>(red));
      if (blue) atomicAdd(&a.stats->blue_wins, static_cast<unsigned long long>(blue));
      if (draws) atomicAdd(&a.stats->draws, static_cast<unsigned long long>(draws));
      if (swaps) atomicAdd(&a.stats->swaps, static_cast<unsigned long long>(swaps));
      if (maxlen) atomicMax(&a.stats->max_length, static_cast<unsigned long long>(maxlen));
    }
  }
}

// (A PAIRED form of this kernel -- two warps per 32 envs, a selector owning header / pegs / selection and an
// evaluator owning links / flags / floods, talking through mailbox words and named barriers -- was built and
// measured in round 2: bit-exact, but 29.2 ms instead of 18.2 ms per launch.  The single warp already runs
// the two chains as instruction-level parallelism; splitting them across warps halved each warp's issue rate
// and added the waits.  profiles/r2_playout_paired_experiment.txt, DESIGN.md section 2.)

int g_num_sms = 0;

#define TW_PLAYOUT_KERNEL playout_kernel
__host__ constexpr size_t launch_smem(int n) {
  return static_cast<size_t>(playout_threads(n)) * playout_words(n) * sizeof(uint32_t) + kSelectLutBytes;
}

template <int NT, bool kTrace>
cudaError_t launch_nt(const PlayoutArgs& a, cudaStream_t s) {
  constexpr int kLaunchThreads = playout_threads(NT), kEnvsPerBlock = playout_threads(NT);
  const size_t smem = launch_smem(NT);
  // persistent grid: as many blocks as fit on the device at once (or fewer for small ranges)
  int per_sm = 0;
  cudaError_t e =
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, TW_PLAYOUT_KERNEL<NT, kTrace>, kLaunchThreads, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  int64_t blocks = (a.count + kEnvsPerBlock - 1) / kEnvsPerBlock;
  const int64_t resident = static_cast<int64_t>(g_num_sms > 0 ? g_num_sms : 148) * per_sm;
  if (blocks > resident) blocks = resident;
  if (TW_PLAYOUT_MAX_BLOCKS > 0 && blocks > TW_PLAYOUT_MAX_BLOCKS) blocks = TW_PLAYOUT_MAX_BLOCKS;
  if (getenv("TWIXT_B200_DEBUG") != nullptr)
    fprintf(stderr, "[twixt_b200] playout n=%d: %lld blocks x %d threads, %zu B smem, %d blocks/SM resident\n", a.n,
            static_cast<long long>(blocks), kLaunchThreads, smem, per_sm);
  TW_PLAYOUT_KERNEL<NT, kTrace><<<static_cast<unsigned>(blocks), kLaunchThreads, smem, s>>>(a);
  return cudaGetLastError();
}

template <int NT, bool kTrace>
cudaError_t setup_one(int n_for_size) {
  const size_t smem = launch_smem(n_for_size);
  if (smem + 1024 > 227 * 1024) return cudaSuccess;  // (an experimental block geometry that does not fit this size: the launch will say so)
  cudaError_t e = cudaFuncSetAttribute(TW_PLAYOUT_KERNEL<NT, kTrace>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem));
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(TW_PLAYOUT_KERNEL<NT, kTrace>, cudaFuncAttributePreferredSharedMemoryCarveout,
                              cudaSharedmemCarveoutMaxShared);
}

template <int NT>
cudaError_t setup_nt(int n_for_size) {
  cudaError_t e = setup_one<NT, false>(n_for_size);
  return e != cudaSuccess ? e : setup_one<NT, true>(n_for_size);
}

template <int NT>
cudaError_t launch_traced_or_not(const PlayoutArgs& a, cudaStream_t s) {
  return a.out_actions != nullptr ? launch_nt<NT, true>(a, s) : launch_nt<NT, false>(a, s);
}

}  // namespace

// This file is compiled once per size GROUP (-DTW_PLAYOUT_GROUP=g, g = 0..4; build.py runs the five
// compilations in parallel): group g holds the kernels specialised for the board sizes 5+g, 10+g, 15+g and
// 20+g, so every board size 5..24 runs with its size fixed at compile time (the run-time-size form of the
// same kernel was 1.3x slower).  twixt_kernels_api.cu dispatches on (n - 5) % 5.
#ifndef TW_PLAYOUT_GROUP
#error "compile with -DTW_PLAYOUT_GROUP=0..4"
#endif
#define TW_CAT2(a, b) a##b
#define TW_CAT(a, b) TW_CAT2(a, b)
constexpr int kGroup = TW_PLAYOUT_GROUP;
static_assert(kGroup >= 0 && kGroup < 5 && TWIXT_MIN_BOARD_SIZE == 5 && TWIXT_MAX_BOARD_SIZE == 24, "size groups");

cudaError_t TW_CAT(playout_setup_g, TW_PLAYOUT_GROUP)() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  if ((e = setup_nt<5 + kGroup>(5 + kGroup)) != cudaSuccess) return e;
  if ((e = setup_nt<10 + kGroup>(10 + kGroup)) != cudaSuccess) return e;
  if ((e = setup_nt<15 + kGroup>(15 + kGroup)) != cudaSuccess) return e;
  return setup_nt<20 + kGroup>(20 + kGroup);
}

cudaError_t TW_CAT(launch_playout_g, TW_PLAYOUT_GROUP)(const PlayoutArgs& a, cudaStream_t s) {
  if (a.count <= 0) return cudaSuccess;
  switch (a.n) {
    case 5 + kGroup: return launch_traced_or_not<5 + kGroup>(a, s);
    case 10 + kGroup: return launch_traced_or_not<10 + kGroup>(a, s);
    case 15 + kGroup: return launch_traced_or_not<15 + kGroup>(a, s);
    case 20 + kGroup: return launch_traced_or_not<20 + kGroup>(a, s);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace twixt
