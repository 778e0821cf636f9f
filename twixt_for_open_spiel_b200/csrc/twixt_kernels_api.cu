// twixt_kernels_api.cu -- the per-call kernels behind the State surface:
// reset (NewInitialState), clone, LegalActions (list + mask), ApplyAction,
// CurrentPlayer / IsTerminal / Returns and ObservationTensor.
//
// All of them are HBM-bound byte/bit work (no tensor cores: nothing here is a
// contraction).  Mapping:
//   reset / clone       one thread per 16-byte piece of a record (128-bit stores)
//   legal list / mask   persistent warps (grid = SMs x occupancy), one env per
//                       warp at a time, lane = board column; popc + ballot
//                       prefix sum places each lane's chunk of the ascending
//                       action list; inputs fetched one env ahead
//   apply / replay      one thread per env working in place on its record
//                       (touches only the few words a move needs)
//   observation(+mask)  persistent blocks, one env per block at a time, record
//                       staged in shared memory one env ahead, float4 stores
//   validate            one warp per imported record, lane = board column
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/twixt_b200.h"
#include "twixt_engine.cuh"
#include "twixt_kernels.cuh"

namespace twixt {

namespace {

constexpr unsigned kFullMask = 0xFFFFFFFFu;
constexpr int kFloodStack = 48;

// Read-only loads of a PART of a record, with the 64-byte L2 fetch-size hint: the kernels below use the
// first 16..208 bytes of each 880-byte record, and the default 128-byte fetch pulled 320 bytes per env out
// of DRAM where 256 do (legal mask: 0.168 -> 0.162 ms per 1 Mi envs).
__device__ __forceinline__ uint4 ldg128(const uint32_t* p) {
  uint4 v;
  asm volatile("ld.global.nc.L2::64B.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ldg32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.global.nc.L2::64B.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// ---------------------------------------------------------------- reset ---
// Board::Board (twixtboard.cc:168-174): empty board, both legal lists full.
__global__ void reset_kernel(uint32_t* __restrict__ records, int64_t count, int n, int quads_per_record) {
  const int64_t total = count * quads_per_record;
  const uint32_t cnt = static_cast<uint32_t>(n * (n - 2));
  for (int64_t q = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; q < total;
       q += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int in_rec = static_cast<int>(q % quads_per_record);
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (in_rec == 0) v = make_uint4(0u, 0u, kNoMove, cnt | (cnt << 16));
    reinterpret_cast<uint4*>(records)[q] = v;
  }
}

// ---------------------------------------------------------------- clone ---
// State::Clone (twixt.h:80-82): dst env i <- src env (src_ids ? src_ids[i] : i).
// Gathered ids are checked HERE (they may live on the device, where the host cannot see them): an id outside
// [0, num_envs) or inside the destination range [dst_first, dst_first + count) copies nothing and is
// reported through stats->bad_clone_index (lowest offending position), like apply reports illegal actions.
__global__ void clone_kernel(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src,
                             const int64_t* __restrict__ src_ids, int64_t count, int quads_per_record,
                             int64_t num_envs, int64_t dst_first, DeviceStats* __restrict__ stats) {
  const int64_t total = count * quads_per_record;
  for (int64_t q = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; q < total;
       q += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t env = q / quads_per_record;
    const int in_rec = static_cast<int>(q - env * quads_per_record);
    int64_t from = env;
    if (src_ids != nullptr) {
      from = src_ids[env];
      if (from < 0 || from >= num_envs || (from >= dst_first && from < dst_first + count)) {
        if (in_rec == 0) atomicMin(&stats->bad_clone_index, static_cast<unsigned int>(env));
        continue;
      }
    }
    reinterpret_cast<uint4*>(dst)[q] = __ldg(reinterpret_cast<const uint4*>(src) + from * quads_per_record + in_rec);
  }
}

// ------------------------------------------------------ legal list / mask ---
// One warp per env at a time, lane = board column, persistent warps striding
// over the env range (a grid of 1 M tiny blocks is bound by block launch rate,
// not by HBM).  The three loads an env needs (header, red word, blue word of
// the lane's column) are independent and are issued one env ahead.
constexpr int kLegalWarps = 8;  // warps per block (mask kernel: 4 / 8 / 16 measured equal)
// the list kernel runs 16 warps per block, 3 blocks per SM: the same 48 resident warps as 8 x 6, measured 2.7 %
// faster (0.2726 -> 0.2650 ms per 1 Mi envs with uint16 actions)
constexpr int kListWarps = 16, kListMinBlocks = 3;

struct LegalInputs {
  uint4 hw;
  uint32_t red, blue;
};

__device__ __forceinline__ LegalInputs legal_fetch(const uint32_t* rec, int n, int lane) {
  LegalInputs in;
  const int col = lane < n ? lane : 0;
  in.hw = ldg128(rec);
  in.red = ldg32(rec + kHeaderWords + col);
  in.blue = ldg32(rec + kHeaderWords + n + col);
  return in;
}

// Legal word of column `lane` (0 for lanes >= n and for terminal envs):
// TwixTState::LegalActions twixt.h:86-90.
__device__ __forceinline__ uint32_t legal_word_of(const LegalInputs& in, int n, int lane) {
  Header h;
  unpack_header(in.hw.x, in.hw.y, in.hw.z, in.hw.w, h);
  if (h.result != kOpen || lane >= n) return 0u;
  const uint32_t play = playable_word(n, static_cast<int>(h.ply & 1u), lane);
  if (h.ply == 1u) return play;
  return play & ~(in.red | in.blue);
}

// The legal cells of an env form one n*n-bit string in action order (action =
// x*n + y is column-major, twixtboard.cc:603-605).  It is cut into 32 equal
// chunks of ceil(n*n/32) <= 18 bits, one per lane, so all 32 lanes carry the
// same load whatever the board size (a chunk spans at most two column words,
// fetched from their lanes by shuffle).  popc + warp prefix sum give every
// chunk its offset in the ascending list; each lane expands its chunk into a
// shared-memory row with a fixed, branch-free run of predicated stores (one
// bit test, one store and one pointer bump per cell: no loop, no divergence
// between lanes with different populations), then the warp streams the row
// out with coalesced 16-byte stores.
constexpr int kMaxChunkBits = (TWIXT_MAX_BOARD_SIZE * TWIXT_MAX_BOARD_SIZE + 31) / 32;
static_assert(kMaxChunkBits < 32, "chunk populations must fit the 5-ballot prefix sum");

// 16 bytes of output (kPerVec = 16 / sizeof(T) actions) from the uint16 staging row, vector index v
template <typename T>
__device__ __forceinline__ uint4 widen_actions(const uint16_t* row, int v);
template <>
__device__ __forceinline__ uint4 widen_actions<uint16_t>(const uint16_t* row, int v) {
  return reinterpret_cast<const uint4*>(row)[v];
}
template <>
__device__ __forceinline__ uint4 widen_actions<int32_t>(const uint16_t* row, int v) {
  const uint2 p = reinterpret_cast<const uint2*>(row)[v];
  return make_uint4(p.x & 0xFFFFu, p.x >> 16, p.y & 0xFFFFu, p.y >> 16);
}
template <>
__device__ __forceinline__ uint4 widen_actions<int64_t>(const uint16_t* row, int v) {
  const uint32_t p = reinterpret_cast<const uint32_t*>(row)[v];
  return make_uint4(p & 0xFFFFu, 0u, p >> 16, 0u);
}

template <typename T>
__global__ void __launch_bounds__(kListWarps * 32, kListMinBlocks) legal_actions_kernel(
    const uint32_t* __restrict__ records, int64_t count, int n, int rw, T* __restrict__ out_actions, int64_t stride,
    int32_t* __restrict__ out_counts) {
  constexpr int kPerVec = 16 / static_cast<int>(sizeof(T));
  // the row is staged as uint16 whatever T is (actions < 576): a quarter of the shared-memory traffic of an
  // int64 row; the copy-out widens kPerVec entries into each 16-byte store
  __shared__ __align__(16) uint16_t rows[kListWarps][TWIXT_MAX_BOARD_SIZE * (TWIXT_MAX_BOARD_SIZE - 2)];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kListWarps;
  int64_t env = blockIdx.x * static_cast<int64_t>(kListWarps) + warp;
  if (env >= count) return;  // whole warp leaves together
  uint16_t* row = rows[warp];
  // this lane's chunk of the flat cell string: cells [first, first + chunk_bits)
  const int cells = n * n;
  const int chunk_bits = (cells + 31) >> 5;
  const int first = lane * chunk_bits;
  const int x0 = min(first / n, n - 1), y0 = first - (first / n) * n;
  const int x1 = min(x0 + 1, n - 1);
  const uint32_t chunk_mask = first >= cells ? 0u : ((1u << min(chunk_bits, cells - first)) - 1u);
  const int64_t rec_step = nwarps * rw;
  const uint32_t* rec = records + env * rw;
  T* dst = out_actions != nullptr ? out_actions + env * stride : nullptr;
  const int64_t dst_step = nwarps * stride;
  // rows start 16-byte aligned for every env iff the base is and the stride is a whole number of vectors
  const bool vec_ok = (reinterpret_cast<uintptr_t>(out_actions) & 15u) == 0 && stride % kPerVec == 0;
  LegalInputs cur = legal_fetch(rec, n, lane);
  for (; env < count; env += nwarps) {
    rec += rec_step;
    LegalInputs nxt = cur;
    if (env + nwarps < count) nxt = legal_fetch(rec, n, lane);
    const uint32_t colw = legal_word_of(cur, n, lane);
    const uint32_t w0 = __shfl_sync(kFullMask, colw, x0), w1 = __shfl_sync(kFullMask, colw, x1);
    const uint32_t w = ((w0 >> y0) | (w1 << (n - y0))) & chunk_mask;
    // prefix sum of the 32 chunk populations (each <= kMaxChunkBits < 32) by ballots, one per bit of the
    // count: shuffles would queue on the shared-memory data pipe, which is what bounds this kernel
    const int c = __popc(w);
    const uint32_t le_mask = 0xFFFFFFFFu >> (31 - lane);
    int incl = 0, total = 0;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const uint32_t bk = __ballot_sync(kFullMask, (c >> k) & 1);
      incl += __popc(bk & le_mask) << k;
      total += __popc(bk) << k;
    }
    if (out_counts != nullptr && lane == 0) out_counts[env] = total;
    if (dst != nullptr) {
      // flat cell index == action; bits past the chunk are zero, so the run needs no length test
      uint16_t* slot = row + (incl - c);
#pragma unroll
      for (int j = 0; j < kMaxChunkBits; ++j) {
        if ((w >> j) & 1u) {
          *slot = static_cast<uint16_t>(first + j);
          ++slot;
        }
      }
      __syncwarp();
      if (vec_ok) {
        const int nvec = total / kPerVec;
#pragma unroll 1
        for (int v = lane; v < nvec; v += 32)
          reinterpret_cast<uint4*>(dst)[v] = widen_actions<T>(row, v);
        const int i = nvec * kPerVec + lane;  // fewer than kPerVec <= 8 entries are left
        if (i < total) dst[i] = static_cast<T>(row[i]);
      } else {
#pragma unroll 1
        for (int i = lane; i < total; i += 32) dst[i] = static_cast<T>(row[i]);
      }
      __syncwarp();  // the row is reused by the next env
      dst += dst_step;
    }
    cur = nxt;
  }
}

// [count, n*n] uint8 mask.  For n % 4 == 0 every lane turns its column word into n mask bytes with the
// nibble-spreading multiply (4 bits -> 4 bytes), the warp stages the n*n bytes in shared memory and
// writes them out with 16-byte stores; other sizes take the byte-wise path.
// kWords = n/4 fixed at compile time for the fast path (0 = byte-wise path for any n).
template <int kWords>
__global__ void __launch_bounds__(kLegalWarps * 32) legal_mask_kernel(const uint32_t* __restrict__ records,
                                                                      int64_t count, int n, int rw,
                                                                      uint8_t* __restrict__ out) {
  __shared__ __align__(16) uint32_t rows[kLegalWarps][TWIXT_MAX_BOARD_SIZE * TWIXT_MAX_BOARD_SIZE / 4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kLegalWarps;
  int64_t env = blockIdx.x * static_cast<int64_t>(kLegalWarps) + warp;
  if (env >= count) return;
  const int cells = n * n;
  uint32_t* row = rows[warp];
  LegalInputs cur = legal_fetch(records + env * rw, n, lane);
  for (; env < count; env += nwarps) {
    const int64_t next = env + nwarps;
    LegalInputs nxt = cur;
    if (next < count) nxt = legal_fetch(records + next * rw, n, lane);
    const uint32_t w = legal_word_of(cur, n, lane);
    uint8_t* dst = out + env * cells;
    if (kWords > 0) {
      if (lane < 4 * kWords) {
#pragma unroll
        for (int q = 0; q < kWords; ++q)  // bits 4q..4q+3 -> one byte each
          row[lane * kWords + q] = (((w >> (4 * q)) & 0xFu) * 0x00204081u) & 0x01010101u;
      }
      __syncwarp();
      constexpr int kVecs = kWords * kWords;  // n*n/16 with n = 4*kWords
#pragma unroll
      for (int v = 0; v < (kVecs + 31) / 32; ++v)
        if (v * 32 + lane < kVecs)
          reinterpret_cast<uint4*>(dst)[v * 32 + lane] = reinterpret_cast<const uint4*>(row)[v * 32 + lane];
      __syncwarp();
    } else {
      for (int base = 0; base < cells; base += 32) {
        const int c = base + lane;
        const int x = min(c / n, n - 1);
        const int y = c - x * n;
        const uint32_t col = __shfl_sync(kFullMask, w, x);
        if (c < cells) dst[c] = static_cast<uint8_t>((col >> y) & 1u);
      }
    }
    cur = nxt;
  }
}

// ---------------------------------------------------------------- apply ---
// TwixTState::DoApplyAction (twixt.h:93-104): legality, Board::ApplyAction,
// turn hand-over (implicit in ply parity / result).
// (the launch bound lets ptxas use 93 registers instead of the 64 its default heuristic stops at: the independent
// loads of link_move stay in flight together, 0.2294 -> 0.2171 ms per 1 Mi envs)
__global__ void __launch_bounds__(128, 1) apply_kernel(uint32_t* __restrict__ records, int64_t count, int n, int rw,
                             const int32_t* __restrict__ actions, int32_t* __restrict__ out_status,
                             DeviceStats* __restrict__ stats) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= count) return;
  const int action = actions[i];
  int status = 2;
  if (action >= 0) {
    RecordRef<1> b{records + i * rw, n};
    const uint4 hw = *reinterpret_cast<const uint4*>(b.p);
    Header h;
    unpack_header(hw.x, hw.y, hw.z, hw.w, h);
    if (!is_legal(b, h, action)) {
      status = 1;
      atomicMin(&stats->illegal_index, static_cast<unsigned int>(i));  // host names this action in its message
    } else {
      const int x = action / n;
      apply_legal_cell<kFloodStack>(b, h, x, action - x * n);
      uint4 o;
      pack_header(h, o.x, o.y, o.z, o.w);
      *reinterpret_cast<uint4*>(b.p) = o;
      status = 0;
    }
  }
  if (out_status != nullptr) out_status[i] = status;
}

// --------------------------------------------------------------- replay ---
// A whole action history per env in ONE launch (upstream serialises a state as its action history and
// deserialises by replaying it, spiel.cc State::Serialize / Game::DeserializeState; here that replay runs on
// the device instead of one apply launch per move).  actions is [count, stride] int32, env i applies
// actions[i*stride + 0 .. len_i) in order from its CURRENT state with the legality test of DoApplyAction
// (twixt.h:93-104); len_i = lengths[i] if given, else the row up to its first negative entry.  An env stops
// at its first illegal action (state as reached so far); out_applied[i] = moves made.
__global__ void __launch_bounds__(128, 1) replay_kernel(uint32_t* __restrict__ records, int64_t count, int n, int rw,
                              const int32_t* __restrict__ actions, int64_t stride, const int32_t* __restrict__ lengths,
                              int32_t* __restrict__ out_applied, DeviceStats* __restrict__ stats) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= count) return;
  RecordRef<1> b{records + i * rw, n};
  const uint4 hw = *reinterpret_cast<const uint4*>(b.p);
  Header h;
  unpack_header(hw.x, hw.y, hw.z, hw.w, h);
  const int32_t* row = actions + i * stride;
  const int64_t len = lengths != nullptr ? static_cast<int64_t>(lengths[i]) : stride;
  int k = 0;
  for (; k < len && k < stride; ++k) {
    const int action = row[k];
    if (action < 0) break;
    if (!is_legal(b, h, action)) {
      // lowest env first; the low word carries the action for the host's message (twixt.h:96)
      atomicMin(&stats->replay_illegal, (static_cast<unsigned long long>(i) << 32) | static_cast<uint32_t>(action));
      break;
    }
    const int x = action / n;
    apply_legal_cell<kFloodStack>(b, h, x, action - x * n);
  }
  uint4 o;
  pack_header(h, o.x, o.y, o.z, o.w);
  *reinterpret_cast<uint4*>(b.p) = o;
  if (out_applied != nullptr) out_applied[i] = k;
}

// ----------------------------------------------------------------- step ---
// twixt_step: one env, one warp, one launch -- (reset |) apply, then everything an unbatched caller asks
// next (twixt.h:38-104): status, CurrentPlayer, IsTerminal, Returns and the ascending LegalActions as int64
// (open_spiel::Action).  The outputs normally live in the batch's pinned, device-mapped arena.
__global__ void __launch_bounds__(32) step_kernel(uint32_t* __restrict__ rec, int n, int rw, int action,
                                                  twixt_step_result* __restrict__ out, int64_t* __restrict__ out_legal) {
  const int lane = threadIdx.x;
  RecordRef<1> b{rec, n};
  int status = 0;
  if (action == TWIXT_STEP_RESET) {
    const uint32_t cnt = static_cast<uint32_t>(n * (n - 2));
    for (int w = lane; w < rw; w += 32) rec[w] = w == 2 ? kNoMove : (w == 3 ? (cnt | (cnt << 16)) : 0u);
  } else if (action >= 0 && lane == 0) {
    Header h0;
    load_header(b, h0);
    if (!is_legal(b, h0, action)) {
      status = 1;
    } else {
      const int x = action / n;
      apply_legal_cell<kFloodStack>(b, h0, x, action - x * n);
      store_header(b, h0);
    }
  }
  __syncwarp();  // lane 0's (or every lane's) record writes are visible to the whole warp
  Header h;
  load_header(b, h);
  const uint32_t w = (lane < n && h.result == kOpen) ? legal_word(b, h, lane) : 0u;
  const int c = __popc(w);
  int incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int up = __shfl_up_sync(kFullMask, incl, o);
    if (lane >= o) incl += up;
  }
  const int total = __shfl_sync(kFullMask, incl, 31);
  if (out_legal != nullptr) {
    int64_t* dst = out_legal + (incl - c);
    uint32_t rest = w;
    while (rest) {  // ascending: column-major, action = x*n + y (twixtboard.cc:603-605)
      const int y = tw_ctz(rest);
      rest &= rest - 1u;
      *dst++ = static_cast<int64_t>(lane * n + y);
    }
  }
  if (lane == 0) {
    out->status = status;
    out->current_player = current_player(h);
    out->is_terminal = h.result != kOpen ? 1 : 0;
    out->num_legal = total;
    const float r = h.result == kRedWin ? 1.0f : (h.result == kBlueWin ? -1.0f : 0.0f);
    out->returns[0] = r;
    out->returns[1] = r == 0.0f ? 0.0f : -r;
  }
}

// ------------------------------------------------------------- validate ---
// twixt_import_state takes records from the caller, and the fused playout kernel reads records with its
// bounds tests deliberately removed (twixt_kernel_playout.cu, PlayoutRef), so what comes in is checked first.
// The reference can only reach a state through DoApplyAction (twixt.h:93-104); these are the invariants
// every reachable record has and every kernel relies on.  One warp per record, lane = board column:
//   header     result/swapped bits only, ply <= n*n-3, swapped => ply >= 2, result != open => ply >= 1
//   rows       no plane has a bit at a row >= n; padding words are zero
//   pegs       red and blue disjoint; red never in column 0 / n-1, blue never in row 0 / n-1
//              (twixtboard.cc:252-276; the corners follow), popc(red) = ceil(ply/2) - swapped, popc(blue) = ply/2
//   first move word 2 = 0xFFFFFFFF iff ply = 0, else a red first move whose peg (or, after a swap, the blue
//              peg on the turned cell, twixtboard.cc:465-475) is on the board
//   links      a link bit sits on a peg whose knight neighbour in that direction holds a peg of the same
//              colour (so link planes are empty in the columns a link cannot start from)
//   flags      border / blocked bits only on pegs
//   counts     word 3 = empty cells red / blue may still play on, recounted
// The lowest failing env and its reason go to stats->invalid_code by one 64-bit atomicMin.
enum : uint32_t {
  kBadHeader = 1, kBadRows = 2, kBadPegs = 3, kBadFirstMove = 4, kBadLinks = 5, kBadFlags = 6, kBadCounts = 7,
  kBadPadding = 8
};

__global__ void __launch_bounds__(256) validate_kernel(const uint32_t* __restrict__ records, int64_t count, int n,
                                                       int rw, DeviceStats* __restrict__ stats) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  for (int64_t env = blockIdx.x * static_cast<int64_t>(blockDim.x >> 5) + (threadIdx.x >> 5); env < count;
       env += nwarps) {
    const uint32_t* rec = records + env * rw;
    const uint4 hw = ldg128(rec);
    const bool on = lane < n;
    uint32_t w[kNumStatePlanes];
#pragma unroll
    for (int p = 0; p < kNumStatePlanes; ++p) w[p] = on ? __ldg(rec + kHeaderWords + p * n + lane) : 0u;
    const int pad = rw - (kHeaderWords + kNumStatePlanes * n);
    const uint32_t padw = lane < pad ? __ldg(rec + kHeaderWords + kNumStatePlanes * n + lane) : 0u;
    uint32_t bad = 0xFFu;
    const auto flag = [&](bool c, uint32_t code) { bad = (c && code < bad) ? code : bad; };
    const uint32_t full = full_rows(n), inner = inner_rows(n);
    const uint32_t red = w[P_RED], blue = w[P_BLUE], occ = red | blue;
    uint32_t off_rows = 0;
#pragma unroll
    for (int p = 0; p < kNumStatePlanes; ++p) off_rows |= w[p] & ~full;
    flag(off_rows != 0u, kBadRows);
    flag(padw != 0u, kBadPadding);
    flag((red & blue) != 0u, kBadPegs);
    flag((lane == 0 || lane == n - 1) && red != 0u, kBadPegs);
    flag((blue & ~inner) != 0u, kBadPegs);
    flag(((w[P_START] | w[P_END] | w[P_BLOCKED]) & ~occ) != 0u, kBadFlags);
    // pegs one and two columns to the east (lanes >= n hold zeros; n <= 24 keeps lane + 2 inside the warp)
    const uint32_t r1 = __shfl_down_sync(kFullMask, red, 1), r2 = __shfl_down_sync(kFullMask, red, 2);
    const uint32_t b1 = __shfl_down_sync(kFullMask, blue, 1), b2 = __shfl_down_sync(kFullMask, blue, 2);
    const uint32_t ok_nne = (red & (r1 >> 2)) | (blue & (b1 >> 2));  // (x+1, y+2)
    const uint32_t ok_ene = (red & (r2 >> 1)) | (blue & (b2 >> 1));  // (x+2, y+1)
    const uint32_t ok_ese = (red & (r2 << 1)) | (blue & (b2 << 1));  // (x+2, y-1)
    const uint32_t ok_sse = (red & (r1 << 2)) | (blue & (b1 << 2));  // (x+1, y-2)
    flag(((w[P_LINK0] & ~ok_nne) | (w[P_LINK0 + 1] & ~ok_ene) | (w[P_LINK0 + 2] & ~ok_ese) |
          (w[P_LINK0 + 3] & ~ok_sse)) != 0u, kBadLinks);
    // recount: empty playable cells (both fit 16 bits: at most n*(n-2) = 528) and pegs per colour
    uint32_t open2 = ((lane >= 1 && lane <= n - 2) ? __popc(full & ~occ) : 0) | ((on ? __popc(inner & ~occ) : 0) << 16);
    uint32_t pegs2 = __popc(red) | (__popc(blue) << 16);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      open2 += __shfl_xor_sync(kFullMask, open2, o);
      pegs2 += __shfl_xor_sync(kFullMask, pegs2, o);
    }
    const uint32_t ply = hw.x, res = hw.y & 3u, swapped = (hw.y >> 2) & 1u;
    flag((hw.y >> 3) != 0u || ply > static_cast<uint32_t>(n * n - 3) || (swapped && ply < 2u) ||
             (res != kOpen && ply == 0u), kBadHeader);
    flag(hw.w != open2, kBadCounts);
    flag(pegs2 != (((ply + 1u) / 2u - swapped) | ((ply / 2u) << 16)), kBadCounts);
    if (ply == 0u) {
      flag(hw.z != kNoMove, kBadFirstMove);
    } else {
      const uint32_t mo = hw.z;
      const int mx = static_cast<int>(mo) / n, my = static_cast<int>(mo) - mx * n;
      const bool in_range = mo < static_cast<uint32_t>(n * n) && mx >= 1 && mx <= n - 2;
      flag(!in_range, kBadFirstMove);
      if (in_range) {
        // the first peg: red on the cell itself, or blue on the cell turned by 90 degrees after a swap
        const int px = swapped ? my : mx, py = swapped ? n - 1 - mx : my;
        const uint32_t pegs = swapped ? blue : red;
        const bool there = __any_sync(kFullMask, lane == px && ((pegs >> py) & 1u));
        flag(!there, kBadFirstMove);
      }
    }
    bad = __reduce_min_sync(kFullMask, bad);
    if (lane == 0 && bad != 0xFFu)
      atomicMin(&stats->invalid_code, (static_cast<unsigned long long>(env) << 8) | bad);
  }
}

// ---------------------------------------------------------------- query ---
// CurrentPlayer twixt.h:38, IsTerminal twixt.h:45-48, Returns twixt.h:50-63.
__global__ void query_kernel(const uint32_t* __restrict__ records, int64_t count, int rw,
                             int8_t* __restrict__ out_player, uint8_t* __restrict__ out_terminal,
                             float* __restrict__ out_returns) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= count) return;
  const uint4 hw = ldg128(records + i * rw);
  Header h;
  unpack_header(hw.x, hw.y, hw.z, hw.w, h);
  if (out_player != nullptr) out_player[i] = static_cast<int8_t>(current_player(h));
  if (out_terminal != nullptr) out_terminal[i] = h.result != kOpen ? 1 : 0;
  if (out_returns != nullptr) {
    const float r = h.result == kRedWin ? 1.0f : (h.result == kBlueWin ? -1.0f : 0.0f);
    reinterpret_cast<float2*>(out_returns)[i] = make_float2(r, r == 0.0f ? 0.0f : -r);
  }
}

// ---------------------------------------------------------- observation ---
// TwixTState::ObservationTensor (twixt.cc:101-132): [12, n, n-2] float32 per
// env, HBM-write bound (25 KB out per 0.9 KB in at n=24).  Persistent blocks
// stride over the envs; the NEXT env's record is fetched into registers while
// the current one is expanded, so HBM latency hides behind the float stores.
// Per env (all from shared memory):
//  (A) the 12 planes as one bit word per OUTPUT row (GetTensorPosition,
//      twixtboard.cc:590-597).  Red planes: output row r is board row n-1-r
//      gathered across the column words -- a bit-matrix transpose, done by one
//      warp per plane in registers (lane = column, five butterfly steps of
//      shuffle + mask, instead of a 22-iteration bit loop per row).  Blue
//      planes: output row r is ONE column word, bit-reversed.
//  (B) the rows concatenated into one flat bit stream of 12*n*(n-2) bits;
//  (C) each thread turns 4 consecutive stream bits into a float4 (4 | 32, so a
//      group never straddles a word) by one 16-entry table look-up.
//
// kMask: the same pass also writes the env's [n*n] uint8 legal-action mask (upstream LegalActionsMask; the
// AlphaZero-style producer of BASELINE config C5 wants both), so the record is read from HBM once for the
// two outputs.  The mask is 576 of the 25 920 output bytes at n = 24.
//
// TW_OBS_BULK = 1 (the default; 0 keeps the float4-store form for the A/B in DESIGN.md): step (C) writes the
// floats into a double-buffered tile in shared memory and ONE thread hands the whole tile (25 KB at n = 24) to
// the copy engine (cp.async.bulk shared -> global, UBLKCP in SASS), so the expansion of env i+1 overlaps the
// store of env i and no store instruction of the SM touches HBM.  Measured at B = 65 536, n = 24:
// observation 0.326 -> 0.312 ms, observation + mask 0.339 -> 0.297 ms (0.79 -> 0.89 of the copy peak).
#ifndef TW_OBS_BULK
#define TW_OBS_BULK 1
#endif
constexpr int kObsThreads = 256;
constexpr int kObsPlaneWords = 12 * TWIXT_MAX_BOARD_SIZE;
constexpr int kObsStreamWords = (12 * TWIXT_MAX_BOARD_SIZE * (TWIXT_MAX_BOARD_SIZE - 2) + 31) / 32;
constexpr int kObsRecordWords = (kHeaderWords + kNumStatePlanes * TWIXT_MAX_BOARD_SIZE + 3) & ~3;  // 220 <= 256 threads
[[maybe_unused]] constexpr int kObsMaxFloats = 12 * TWIXT_MAX_BOARD_SIZE * (TWIXT_MAX_BOARD_SIZE - 2);

// 32 x 32 bit-matrix transpose across a warp: lane i holds row i on entry and column i on return.
__device__ __forceinline__ uint32_t warp_transpose32(uint32_t x, int lane) {
#pragma unroll
  for (int j = 16; j >= 1; j >>= 1) {
    const uint32_t m = j == 16 ? 0x0000FFFFu : j == 8 ? 0x00FF00FFu : j == 4 ? 0x0F0F0F0Fu : j == 2 ? 0x33333333u : 0x55555555u;
    const uint32_t other = __shfl_xor_sync(kFullMask, x, j);
    const bool upper = (lane & j) != 0;
    const uint32_t lo = upper ? (other >> j) : x;   // what ends up under the mask
    const uint32_t hi = upper ? x : (other << j);   // ... and outside it
    x = (lo & m) | (hi & ~m);
  }
  return x;
}

template <bool kVec4, bool kMask>
__global__ void __launch_bounds__(kObsThreads, TW_OBS_BULK ? 4 : 8) observation_kernel(
    const uint32_t* __restrict__ records, int64_t count, int n, int rw, float* __restrict__ out,
    uint8_t* __restrict__ out_mask) {
  __shared__ __align__(16) uint32_t rec[kObsRecordWords];  // the env's record
  __shared__ uint32_t rowbits[kObsPlaneWords];             // [12][n] output rows, bit c = tensor column c
  __shared__ uint32_t stream[kObsStreamWords];             // the tensor as a bit stream, output order
  __shared__ uint32_t legalw[TWIXT_MAX_BOARD_SIZE];        // kMask: legal cells per column
  __shared__ __align__(16) float4 lut[16];                 // 4 stream bits -> 4 floats
#if TW_OBS_BULK
  extern __shared__ __align__(128) float tile[];           // [2][total] staged output, double-buffered
#endif
  const int w = n - 2;
  const int rows = 12 * n;
  const int total = rows * w;
  const int stream_words = (total + 31) >> 5;
  const uint32_t wmask = (1u << w) - 1u;
  // bit / w by multiply-shift: m = ceil(2^20 / w) is exact while x * (m*w - 2^20) < 2^20, i.e. for every
  // x < 6336 + 32 and w <= 22; x*m < 2^32 as well (host-checked exhaustively in tests/test_abi.py)
  const uint32_t m_row = ((1u << 20) + w - 1) / w;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 16)
    lut[tid] = make_float4((tid & 1) ? 1.0f : 0.0f, (tid & 2) ? 1.0f : 0.0f, (tid & 4) ? 1.0f : 0.0f,
                           (tid & 8) ? 1.0f : 0.0f);
  int64_t env = blockIdx.x;
  uint32_t pre = (env < count && tid < rw) ? __ldg(records + env * rw + tid) : 0u;
#if TW_OBS_BULK
  int buf = 0;
#endif
  for (; env < count; env += gridDim.x) {
    if (tid < rw) rec[tid] = pre;
    __syncthreads();
    const int64_t next = env + gridDim.x;
    if (next < count && tid < rw) pre = __ldg(records + next * rw + tid);  // in flight during the expansion
    RecordRef<1> b{rec, n};
    // ---- (A) one bit word per output row
    if (warp < 6) {
      // red plane p = warp: lane = board column x; after the transpose lane = board row y, bit = column x
      const uint32_t colw = lane < n ? obs_plane_word(b, warp, lane) : 0u;
      const uint32_t roww = warp_transpose32(colw, lane);
      if (lane < n) rowbits[warp * n + (n - 1 - lane)] = (roww >> 1) & wmask;  // (r, c) <- cell (c+1, n-1-r)
    }
    {
      // blue planes: (r, c) <- cell (n-1-r, n-2-c): rows 1..n-2 of one column word, reversed.  One word per
      // thread, taken from the top of the block so that the warps busy with a transpose get the fewest.
      const int t = kObsThreads - 1 - tid;
      if (t < 6 * n) {
        const int p = t / n, x = t - p * n;
        rowbits[(6 + p) * n + (n - 1 - x)] = (__brev(obs_plane_word(b, 6 + p, x)) >> (32 - (n - 1))) & wmask;
      }
      if (kMask && tid < n) {  // TwixTState::LegalActions (twixt.h:86-90) as a bit word per column
        Header h;
        unpack_header(rec[0], rec[1], rec[2], rec[3], h);
        legalw[tid] = h.result != kOpen ? 0u : legal_word(b, h, tid);
      }
    }
    __syncthreads();
    // ---- (B) the flat bit stream (+ the legal mask)
    for (int k = tid; k < stream_words; k += kObsThreads) {
      // stream bits [32k, 32k+32): the tail of one row and the heads of the following ones
      const int bit0 = k << 5;
      int row = static_cast<int>((static_cast<uint32_t>(bit0) * m_row) >> 20);
      int have = 0;
      uint32_t acc = 0;
      int off = bit0 - row * w;  // bits of `row` already consumed by earlier words
      while (have < 32 && row < rows) {
        acc |= (rowbits[row] >> off) << have;
        have += w - off;
        off = 0;
        ++row;
      }
      stream[k] = acc;
    }
    if (kMask) {
      const int cells = n * n;
      uint8_t* mdst = out_mask + env * static_cast<int64_t>(cells);
      if ((cells & 3) == 0 && (reinterpret_cast<uintptr_t>(out_mask) & 3u) == 0) {
        for (int q = tid; q < (cells >> 2); q += kObsThreads) {  // four consecutive cells -> one 4-byte store
          int x = (4 * q) / n, y = 4 * q - x * n;
          uint32_t v = 0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            v |= ((legalw[x] >> y) & 1u) << (8 * j);
            if (++y == n) { y = 0; ++x; }
          }
          reinterpret_cast<uint32_t*>(mdst)[q] = v;
        }
      } else {
        for (int c = tid; c < cells; c += kObsThreads) {
          const int x = c / n;
          mdst[c] = static_cast<uint8_t>((legalw[x] >> (c - x * n)) & 1u);
        }
      }
    }
    __syncthreads();
    // ---- (C) bits -> floats
    float* dst = out + env * static_cast<int64_t>(total);
#if TW_OBS_BULK
    if (kVec4) {
      // the copy engine may still be READING this buffer for the env two iterations back
      if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      __syncthreads();
      float4* t4 = reinterpret_cast<float4*>(tile + buf * kObsMaxFloats);
      for (int q = tid; q < (total >> 2); q += kObsThreads)
        t4[q] = lut[(stream[q >> 3] >> ((q & 7) << 2)) & 15u];
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the copy engine
      __syncthreads();
      if (tid == 0) {
        const uint32_t src = static_cast<uint32_t>(__cvta_generic_to_shared(t4));
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src),
                     "r"(static_cast<uint32_t>(total * 4))
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      buf ^= 1;
      continue;
    }
#endif
    if (kVec4) {
      for (int q = tid; q < (total >> 2); q += kObsThreads)  // total % 4 == 0
        reinterpret_cast<float4*>(dst)[q] = lut[(stream[q >> 3] >> ((q & 7) << 2)) & 15u];
    } else {
      for (int j = tid; j < total; j += kObsThreads) dst[j] = ((stream[j >> 5] >> (j & 31)) & 1u) ? 1.0f : 0.0f;
    }
    // the next iteration's first barrier orders these reads before rec/rowbits/stream are rewritten
  }
#if TW_OBS_BULK
  if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // the tiles must outlive their copies
#endif
}

inline int grid_for(int64_t items, int threads, int max_blocks = 148 * 64) {
  int64_t blocks = (items + threads - 1) / threads;
  if (blocks < 1) blocks = 1;
  if (blocks > max_blocks) blocks = max_blocks;
  return static_cast<int>(blocks);
}

// Grid of a persistent kernel: exactly the blocks that are resident at once (SM count x occupancy), capped by
// the work.  Every block then strides over the same share of the envs; a grid larger than one resident wave
// would leave the last, partly filled wave running alone.
template <typename Kernel>
inline unsigned persistent_grid(Kernel kernel, int threads, int64_t items_per_block_pass, int64_t items) {
  int dev = 0, sms = 148, per_sm = 1;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) {
    (void)cudaGetLastError();
    per_sm = 1;
  }
  return static_cast<unsigned>(grid_for(items, static_cast<int>(items_per_block_pass), sms * per_sm));
}

}  // namespace

cudaError_t launch_reset(uint32_t* records, int64_t count, int n, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int quads = record_words(n) / 4;
  reset_kernel<<<grid_for(count * quads, 256), 256, 0, s>>>(records, count, n, quads);
  return cudaGetLastError();
}

cudaError_t launch_clone(uint32_t* dst, const uint32_t* src, const int64_t* src_ids, int64_t count, int n,
                         int64_t num_envs, int64_t dst_first, DeviceStats* stats, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int quads = record_words(n) / 4;
  clone_kernel<<<grid_for(count * quads, 256), 256, 0, s>>>(dst, src, src_ids, count, quads, num_envs, dst_first,
                                                           stats);
  return cudaGetLastError();
}

cudaError_t launch_legal_actions(const uint32_t* records, int64_t count, int n, void* out_actions, int elem_bytes,
                                 int64_t stride, int32_t* out_counts, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int threads = kListWarps * 32;
  const int rw = record_words(n);
  if (elem_bytes == 2) {
    const auto k = legal_actions_kernel<uint16_t>;
    k<<<persistent_grid(k, threads, kListWarps, count), threads, 0, s>>>(
        records, count, n, rw, static_cast<uint16_t*>(out_actions), stride, out_counts);
  } else if (elem_bytes == 4) {
    const auto k = legal_actions_kernel<int32_t>;
    k<<<persistent_grid(k, threads, kListWarps, count), threads, 0, s>>>(
        records, count, n, rw, static_cast<int32_t*>(out_actions), stride, out_counts);
  } else {
    const auto k = legal_actions_kernel<int64_t>;
    k<<<persistent_grid(k, threads, kListWarps, count), threads, 0, s>>>(
        records, count, n, rw, static_cast<int64_t*>(out_actions), stride, out_counts);
  }
  return cudaGetLastError();
}

cudaError_t launch_legal_mask(const uint32_t* records, int64_t count, int n, uint8_t* out, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int threads = kLegalWarps * 32;
  // the fast path needs word-aligned columns (n % 4 == 0) and 16-byte aligned rows (n*n % 16 == 0 then)
  const bool fast = (n % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15u) == 0);
  const int rw = record_words(n);
  const auto go = [&](auto kernel) {
    kernel<<<persistent_grid(kernel, threads, kLegalWarps, count), threads, 0, s>>>(records, count, n, rw, out);
  };
  switch (fast ? n / 4 : 0) {
    case 2: go(legal_mask_kernel<2>); break;
    case 3: go(legal_mask_kernel<3>); break;
    case 4: go(legal_mask_kernel<4>); break;
    case 5: go(legal_mask_kernel<5>); break;
    case 6: go(legal_mask_kernel<6>); break;
    default: go(legal_mask_kernel<0>); break;
  }
  return cudaGetLastError();
}

cudaError_t launch_apply(uint32_t* records, int64_t count, int n, const int32_t* actions, int32_t* out_status,
                         DeviceStats* stats, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int threads = 128;
  const int64_t blocks = (count + threads - 1) / threads;
  apply_kernel<<<static_cast<unsigned>(blocks), threads, 0, s>>>(records, count, n, record_words(n), actions,
                                                                 out_status, stats);
  return cudaGetLastError();
}

cudaError_t launch_replay(uint32_t* records, int64_t count, int n, const int32_t* actions, int64_t stride,
                          const int32_t* lengths, int32_t* out_applied, DeviceStats* stats, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int threads = 128;
  const int64_t blocks = (count + threads - 1) / threads;
  replay_kernel<<<static_cast<unsigned>(blocks), threads, 0, s>>>(records, count, n, record_words(n), actions, stride,
                                                                  lengths, out_applied, stats);
  return cudaGetLastError();
}

cudaError_t launch_step(uint32_t* record, int n, int action, twixt_step_result* out, int64_t* out_legal, cudaStream_t s) {
  step_kernel<<<1, 32, 0, s>>>(record, n, record_words(n), action, out, out_legal);
  return cudaGetLastError();
}

cudaError_t launch_validate(const uint32_t* records, int64_t count, int n, DeviceStats* stats, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  validate_kernel<<<grid_for(count, 8, 148 * 16), 256, 0, s>>>(records, count, n, record_words(n), stats);
  return cudaGetLastError();
}

const char* invalid_reason_text(unsigned code) {
  switch (code) {
    case kBadHeader: return "header (ply / result / swapped) out of range";
    case kBadRows: return "a plane has bits at rows >= board_size";
    case kBadPegs: return "pegs overlap, stand on a foreign border line, or their number does not fit the ply";
    case kBadFirstMove: return "first-move word does not match the board";
    case kBadLinks: return "a link bit has no same-colour pegs at both ends";
    case kBadFlags: return "border / blocked flags on an empty cell";
    case kBadCounts: return "peg or empty-cell counts do not match the planes";
    case kBadPadding: return "padding words are not zero";
    default: return "unknown";
  }
}

cudaError_t launch_query(const uint32_t* records, int64_t count, int n, int8_t* out_player, uint8_t* out_terminal,
                         float* out_returns, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int threads = 256;
  const int64_t blocks = (count + threads - 1) / threads;
  query_kernel<<<static_cast<unsigned>(blocks), threads, 0, s>>>(records, count, record_words(n), out_player,
                                                                 out_terminal, out_returns);
  return cudaGetLastError();
}

cudaError_t launch_observation(const uint32_t* records, int64_t count, int n, float* out, uint8_t* out_mask,
                               cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int rw = record_words(n);
  const bool vec = (reinterpret_cast<uintptr_t>(out) & 15u) == 0;
  const auto go = [&](auto k) {
#if TW_OBS_BULK
    const size_t tile_bytes = 2 * static_cast<size_t>(kObsMaxFloats) * sizeof(float);
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tile_bytes));
    int dev = 0, sms = 148, per_sm = 1;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, kObsThreads, tile_bytes) != cudaSuccess || per_sm < 1)
      per_sm = 1;
    k<<<grid_for(count, 1, sms * per_sm), kObsThreads, tile_bytes, s>>>(records, count, n, rw, out, out_mask);
#else
    k<<<persistent_grid(k, kObsThreads, 1, count), kObsThreads, 0, s>>>(records, count, n, rw, out, out_mask);
#endif
  };
  if (out_mask != nullptr) {
    if (vec) go(observation_kernel<true, true>);
    else go(observation_kernel<false, true>);
  } else {
    if (vec) go(observation_kernel<true, false>);
    else go(observation_kernel<false, false>);
  }
  return cudaGetLastError();
}

// ------------------------------------------------------ blocked derivation ---
// Runs right after the fused playout kernel on the same records: ORs into P_BLOCKED the bits of every knight pair
// the launch formed (derive_blocked_word), which the kernel's moves no longer write.  The kernel leaves, per env,
// the starting ply clamped to 2 and -- for ply >= 2 -- the cells occupied at the start (PlayoutArgs::start):
//   0  the board was empty, so P_BLOCKED was zero: the derived plane is stored as it is
//   1  one red peg, no pair yet: every pair is new, the derived bits are OR-ed into the plane
//   2  only pairs with a peg on a cell that was empty at the start are counted (a record built by hand may hold
//      an unlinked pair without its bit, which the per-move rules never examine and so never set)
// HBM-bound: one warp per kDeriveEnvs envs reads their peg and link planes (6n words each, the span right after the
// header) with 16-byte loads into shared memory, then lane = column forms the words; the plane is only read back
// for envs that did not start empty.
constexpr int kDeriveWarps = 8, kDeriveEnvs = 4;
constexpr int kDeriveQuads = (6 * TWIXT_MAX_BOARD_SIZE + 3) / 4;  // per env: RED, BLUE, LINK0..3
constexpr int kDeriveLoads = (kDeriveEnvs * kDeriveQuads + 31) / 32;

__global__ void __launch_bounds__(kDeriveWarps * 32) derive_blocked_kernel(uint32_t* __restrict__ records,
                                                                           int64_t count, int n, int rw,
                                                                           const uint32_t* __restrict__ start) {
  __shared__ uint4 planes[kDeriveWarps][kDeriveEnvs * kDeriveQuads];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t first = (blockIdx.x * static_cast<int64_t>(kDeriveWarps) + warp) * kDeriveEnvs;
  if (first >= count) return;  // whole warp leaves together
  const int envs = count - first < kDeriveEnvs ? static_cast<int>(count - first) : kDeriveEnvs;
  const int quads = (6 * n + 3) / 4;  // the span may end inside P_START (odd n): those words are not used
  uint32_t* const rec0 = records + first * rw;
  // every load of the group first, then the shared-memory stores
  uint4 v[kDeriveLoads];
  const uint32_t mode = lane < envs ? start[first + lane] : 0u;
#pragma unroll
  for (int j = 0; j < kDeriveLoads; ++j) {
    const int i = lane + 32 * j, e = i / quads;
    if (e < envs) v[j] = __ldg(reinterpret_cast<const uint4*>(rec0 + e * rw + kHeaderWords) + (i - e * quads));
  }
  // the plane words and start cells of the envs that did not start empty, requested together (one round trip)
  const int x = lane;
  const bool on = x < n;
  uint32_t old[kDeriveEnvs], occ[kDeriveEnvs];
#pragma unroll
  for (int e = 0; e < kDeriveEnvs; ++e) {
    const uint32_t m = __shfl_sync(kFullMask, mode, e);  // warp-uniform
    old[e] = (e < envs && m != 0u && on) ? rec0[e * rw + kHeaderWords + P_BLOCKED * n + x] : 0u;
    occ[e] = (e < envs && m == 2u && on) ? start[count + (first + e) * n + x] : 0u;
  }
  uint32_t* const sw = reinterpret_cast<uint32_t*>(planes[warp]);
#pragma unroll
  for (int j = 0; j < kDeriveLoads; ++j) {
    const int i = lane + 32 * j, e = i / quads;
    if (e < envs) reinterpret_cast<uint4*>(sw + e * 4 * quads)[i - e * quads] = v[j];
  }
  __syncwarp();
#pragma unroll
  for (int e = 0; e < kDeriveEnvs; ++e) {
    if (e >= envs) break;  // warp-uniform
    const uint32_t* s = sw + e * 4 * quads;
    const uint32_t occ1 = __shfl_down_sync(kFullMask, occ[e], 1), occ2 = __shfl_down_sync(kFullMask, occ[e], 2);
    uint32_t bits = 0u;
#pragma unroll
    for (int c = 0; c < 2; ++c) {  // P_RED, P_BLUE
      const uint32_t p0 = on ? s[c * n + x] : 0u, p1 = x + 1 < n ? s[c * n + x + 1] : 0u;
      const uint32_t p2 = x + 2 < n ? s[c * n + x + 2] : 0u;
      const uint32_t link[4] = {on ? s[(P_LINK0 + 0) * n + x] : 0u, on ? s[(P_LINK0 + 1) * n + x] : 0u,
                                on ? s[(P_LINK0 + 2) * n + x] : 0u, on ? s[(P_LINK0 + 3) * n + x] : 0u};
      bits |= derive_blocked_word(p0, p1, p2, p0 & ~occ[e], p1 & ~occ1, p2 & ~occ2, link);
    }
    if (on) rec0[e * rw + kHeaderWords + P_BLOCKED * n + x] = old[e] | bits;
  }
}

cudaError_t launch_derive_blocked(uint32_t* records, int64_t count, int n, const uint32_t* start, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int64_t blocks = (count + kDeriveWarps * kDeriveEnvs - 1) / (kDeriveWarps * kDeriveEnvs);
  derive_blocked_kernel<<<static_cast<unsigned>(blocks), kDeriveWarps * 32, 0, s>>>(records, count, n,
                                                                                      record_words(n), start);
  return cudaGetLastError();
}

// The fused playout kernel: one compiled form per board size, in five translation units (size groups).
cudaError_t playout_setup() {
  cudaError_t e;
  if ((e = playout_setup_g0()) != cudaSuccess) return e;
  if ((e = playout_setup_g1()) != cudaSuccess) return e;
  if ((e = playout_setup_g2()) != cudaSuccess) return e;
  if ((e = playout_setup_g3()) != cudaSuccess) return e;
  return playout_setup_g4();
}

cudaError_t launch_playout(const PlayoutArgs& a, cudaStream_t s) {
  if (a.n < TWIXT_MIN_BOARD_SIZE || a.n > TWIXT_MAX_BOARD_SIZE) return cudaErrorInvalidValue;
  cudaError_t e;
  switch ((a.n - TWIXT_MIN_BOARD_SIZE) % 5) {
    case 0: e = launch_playout_g0(a, s); break;
    case 1: e = launch_playout_g1(a, s); break;
    case 2: e = launch_playout_g2(a, s); break;
    case 3: e = launch_playout_g3(a, s); break;
    default: e = launch_playout_g4(a, s); break;
  }
  if (e != cudaSuccess || a.start == nullptr || a.n < kPlayoutDeriveMinN) return e;
  return launch_derive_blocked(a.records, a.count, a.n, a.start, s);
}

}  // namespace twixt
