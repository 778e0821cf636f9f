// twixt_mcts.cu -- kernels of the batched MCTS search (twixt_mcts_* in include/twixt_b200.h).
//
// One warp per tree in every kernel.  A simulation is three launches:
//   mcts_select_kernel   descend from the root (warp-wide argmax over a node's edges, ballot/popc for the
//                        unvisited-edge draw), expand a node on its second visit, create the child that a
//                        simulation first reaches, and write the leaf record to its evaluator: R rollout slots
//                        (built-in evaluator) or a batch env (stepwise form)
//   launch_playout       the EXISTING fused playout kernel over the rollout slots, with the stream ids the
//                        select kernel wrote (twixt_kernel_playout.cu, unchanged; without the blocked-plane
//                        pass of twixt_playout, since only the returns of a rollout are read)
//   mcts_backup_kernel   the leaf value (mean rollout return, caller's value or terminal Returns()) added to
//                        every edge on the path, lanes over the path; a PUCT search expands the leaf here, a
//                        solver search proves nodes up the path from a terminal leaf
// A PUCT search (a.edge_p != nullptr) scores every edge with its prior from the first visit on (no unvisited-edge
// draw) and expands a non-terminal leaf in the backup kernel, where the caller's priors for it are known.
// A solver search (a.root_out != nullptr, MCTS-Solver) keeps an outcome code per edge and per root: a proven child
// is scored by its outcome, and a tree whose root is proven is finished and takes no further part.
// The select and backup kernels are templates on the search kind; the kernels that run once per search or per move
// (begin, root stats, advance, ...) are one kernel each and test the arena's optional arrays for nullptr.
// The scalar arithmetic (scores, draw, tie keys, stream ids, best child) is in twixt_mcts.cuh, shared with the
// host harnesses that check it without a GPU.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/twixt_b200.h"
#include "twixt_engine.cuh"
#include "twixt_kernels.cuh"
#include "twixt_mcts.cuh"

namespace twixt {

namespace {

constexpr unsigned kFullMask = 0xFFFFFFFFu;
constexpr int kMctsFloodStack = 48;  // as the apply kernel
constexpr int kMctsWarps = 4;        // trees per block

__device__ __forceinline__ int64_t mcts_slot(const MctsArena& a, int64_t t, int local) {
  return t * a.S + local;
}

// copy one record (rw is a multiple of 4 words) with 16-byte loads and stores, lanes over the quads
__device__ __forceinline__ void warp_copy_record(uint32_t* dst, const uint32_t* src, int rw, int lane) {
  for (int q = lane; q < rw / 4; q += 32)
    reinterpret_cast<uint4*>(dst)[q] = reinterpret_cast<const uint4*>(src)[q];
}

// Expands node slot g (record rec, header h): the ascending legal list from the column words (lane = column),
// every edge N = 0, W = 0, no child.  Returns the edge count L, also stored as the node's.
__device__ __forceinline__ int warp_expand(const MctsArena& a, int64_t g, const uint32_t* rec, const Header& h, int lane) {
  const int n = a.n;
  const int64_t e0 = g * a.M;
  RecordRef<1> b{const_cast<uint32_t*>(rec), n};
  const uint32_t w = lane < n ? legal_word(b, h, lane) : 0u;
  const int c = __popc(w);
  int incl = c;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int o = __shfl_up_sync(kFullMask, incl, d);
    if (lane >= d) incl += o;
  }
  const int legal = __shfl_sync(kFullMask, incl, 31);
  uint32_t rest = w;
  for (int i = incl - c; rest != 0u; ++i) {
    const int y = __ffs(static_cast<int>(rest)) - 1;
    rest &= rest - 1u;
    a.edge_action[e0 + i] = static_cast<uint16_t>(lane * n + y);
  }
  for (int i = lane; i < legal; i += 32) {
    a.edge_n[e0 + i] = 0u;
    a.edge_w[e0 + i] = 0.0;
    a.edge_child[e0 + i] = -1;
  }
  if (lane == 0) a.node_legal[g] = legal;
  __syncwarp();
  return legal;
}

// ----------------------------------------------------------------- begin ---
// The root of tree t is a COPY of env roots + t; every tree is cleared to its root alone (a solver search: and its
// root code to unproven; K > 1: its V(s) to 0).  The node count goes to tree entry t*K, and K = 1 without virtual
// visits.
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_begin_kernel(MctsArena a, const uint32_t* __restrict__ roots,
                                                                     int64_t count) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int64_t root = mcts_slot(a, t, 0);
  warp_copy_record(a.node_rec + root * a.rw, roots + t * a.rw, a.rw, lane);
  if (lane == 0) {
    a.node_legal[root] = -1;
    a.node_n[root] = 0u;
    if (a.node_v != nullptr) a.node_v[root] = 0;
    a.tree[t * a.K] = make_int4(1, 0, 0, kLeafNeedsValue);
    if (a.root_out != nullptr) a.root_out[t] = 0;
  }
}

// ------------------------------------------------------- select, K > 1 ---
// The K descents of tree t in a search with K = a.K > 1 leaves per step (the kVirtual select kernels): descent j
// is simulation k + j, scores with the virtual counts of descents 0 .. j-1 (n_eff, N_eff(s), w_eff: twixt_mcts.cuh),
// writes leaf row t*K + j (tree entry, status, leaf env or its R rollout slots), then adds V += 1 along its path
// (lanes over the path) and on its leaf.  The descent itself is the one of the kernel below.
template <bool kPuct>
__device__ __forceinline__ void select_descents(const MctsArena& a, int64_t t, int lane, uint64_t seed, uint32_t T,
                                                uint32_t k, double uct_c, uint32_t* __restrict__ leaf_dst,
                                                int32_t* __restrict__ out_status) {
  const int n = a.n, rw = a.rw, K = a.K;
  int nodes = a.tree[t * K].x;
  for (int j = 0; j < K; ++j) {
    const int64_t row = t * K + j;
    int2* path = a.path + row * a.P;
    int node = 0, depth = 0;
    bool terminal;
    for (;;) {
      const int64_t g = mcts_slot(a, t, node);
      uint32_t* rec = a.node_rec + g * rw;
      const uint4 hw = *reinterpret_cast<const uint4*>(rec);
      Header h;
      unpack_header(hw.x, hw.y, hw.z, hw.w, h);
      terminal = h.result != kOpen;
      const uint32_t visits = a.node_n[g];
      if (terminal || visits == 0u) break;
      const uint32_t visits_eff = visits + a.node_v[g];
      const int64_t e0 = g * a.M;
      int legal = a.node_legal[g];
      int edge;
      if constexpr (kPuct) {
        const double sq = mcts_sqrt_visits(visits_eff);
        double best = 0.0;
        uint32_t bk = 0u;
        int bi = 0x7FFFFFFF;
        for (int i = lane; i < legal; i += 32) {
          const uint8_t o = a.edge_out[e0 + i];
          const uint32_t v = a.edge_v[e0 + i];
          const double sc = o != 0 ? static_cast<double>(mcts_outcome_value(o))
                                   : mcts_puct_score(mcts_virtual_w(a.edge_w[e0 + i], v, a.vl), a.edge_n[e0 + i] + v,
                                                     a.edge_p[e0 + i], sq, uct_c);
          const uint32_t key = a.edge_key[e0 + i];
          if (bi == 0x7FFFFFFF || mcts_puct_beats(sc, key, i, best, bk, bi)) {
            best = sc;
            bk = key;
            bi = i;
          }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
          const double os = __shfl_xor_sync(kFullMask, best, d);
          const uint32_t ok = __shfl_xor_sync(kFullMask, bk, d);
          const int oi = __shfl_xor_sync(kFullMask, bi, d);
          if (oi != 0x7FFFFFFF && (bi == 0x7FFFFFFF || mcts_puct_beats(os, ok, oi, best, bk, bi))) {
            best = os;
            bk = ok;
            bi = oi;
          }
        }
        edge = bi;
      } else {
        if (legal < 0) {
          legal = warp_expand(a, g, rec, h, lane);
          for (int i = lane; i < legal; i += 32) a.edge_v[e0 + i] = 0;
          __syncwarp();
        }
        // edges with n_eff == 0
        int unvisited = 0;
        for (int i = lane; i < legal; i += 32) unvisited += a.edge_n[e0 + i] + a.edge_v[e0 + i] == 0u ? 1 : 0;
        unvisited = __reduce_add_sync(kFullMask, unvisited);
        if (unvisited > 0) {
          int pick = static_cast<int>(mcts_draw(seed, T, k + static_cast<uint32_t>(j), static_cast<uint32_t>(unvisited)));
          edge = -1;
          for (int base = 0; edge < 0; base += 32) {
            const int i = base + lane;
            const uint32_t m = __ballot_sync(kFullMask, i < legal && a.edge_n[e0 + i] + a.edge_v[e0 + i] == 0u);
            const int c = __popc(m);
            if (pick < c) edge = base + select_bit(m, pick);
            else pick -= c;
          }
        } else {
          const double log_parent = a.log_table[visits_eff];
          double best = 0.0;
          int bi = 0x7FFFFFFF;
          for (int i = lane; i < legal; i += 32) {
            const uint32_t v = a.edge_v[e0 + i];
            const double sc = mcts_uct_score(mcts_virtual_w(a.edge_w[e0 + i], v, a.vl), a.edge_n[e0 + i] + v,
                                             log_parent, uct_c);
            if (bi == 0x7FFFFFFF || mcts_score_beats(sc, i, best, bi)) {
              best = sc;
              bi = i;
            }
          }
#pragma unroll
          for (int d = 16; d > 0; d >>= 1) {
            const double os = __shfl_xor_sync(kFullMask, best, d);
            const int oi = __shfl_xor_sync(kFullMask, bi, d);
            if (oi != 0x7FFFFFFF && (bi == 0x7FFFFFFF || mcts_score_beats(os, oi, best, bi))) {
              best = os;
              bi = oi;
            }
          }
          edge = bi;
        }
      }
      if (lane == 0) path[depth] = make_int2(node, (edge << 1) | static_cast<int>(h.ply & 1u));
      ++depth;
      int child = a.edge_child[e0 + edge];
      if (child < 0) {
        child = nodes++;
        const int64_t gc = mcts_slot(a, t, child);
        uint32_t* crec = a.node_rec + gc * rw;
        warp_copy_record(crec, rec, rw, lane);
        __syncwarp();
        if (lane == 0) {
          RecordRef<1> cb{crec, n};
          Header ch = h;
          const int action = a.edge_action[e0 + edge];
          const int x = action / n;
          apply_legal_cell<kMctsFloodStack>(cb, ch, x, action - x * n);
          uint4 o;
          pack_header(ch, o.x, o.y, o.z, o.w);
          *reinterpret_cast<uint4*>(crec) = o;
          a.node_legal[gc] = -1;
          a.node_n[gc] = 0u;
          a.node_v[gc] = 0;
          a.edge_child[e0 + edge] = child;
          if (kPuct && ch.result != kOpen) a.edge_out[e0 + edge] = mcts_outcome_code(ch, static_cast<int>(h.ply & 1u));
        }
        __syncwarp();
      }
      node = child;
    }
    const uint32_t* leaf = a.node_rec + mcts_slot(a, t, node) * rw;
    if (leaf_dst != nullptr) {
      warp_copy_record(leaf_dst + row * rw, leaf, rw, lane);
    } else {
      for (int r = 0; r < a.R; ++r) warp_copy_record(a.roll_rec + (row * a.R + r) * rw, leaf, rw, lane);
      for (int r = lane; r < a.R; r += 32)
        a.roll_ids[row * a.R + r] = mcts_rollout_stream(T, k + static_cast<uint32_t>(j), static_cast<uint32_t>(a.R),
                                                        static_cast<uint32_t>(r));
    }
    const int status = terminal ? kLeafTerminal : kLeafNeedsValue;
    if (lane == 0) {
      a.tree[row] = make_int4(nodes, node, depth, status);
      if (out_status != nullptr) out_status[row] = status;
    }
    // V += 1 along the path and on the leaf, seen by the next descent
    __syncwarp();
    for (int i = lane; i < depth; i += 32) {
      const int2 p = path[i];
      const int64_t g = mcts_slot(a, t, p.x);
      a.node_v[g] += 1;
      a.edge_v[g * a.M + (p.y >> 1)] += 1;
    }
    if (lane == 0) a.node_v[mcts_slot(a, t, node)] += 1;
    __syncwarp();
  }
  if (lane == 0) a.tree[t * K].x = nodes;  // the node count of the tree
}

// ---------------------------------------------------------------- select ---
// kPuct = (a.edge_p != nullptr), kSolve = (a.root_out != nullptr): one instantiation per search kind, so the UCT
// kernel carries no PUCT code and neither carries solver code.  A solver search's finished tree (proven root) takes
// no path: status kLeafSolved, its leaf env is not written, and in run mode its rollout slots get a copy of the
// root marked drawn, which the playout kernel counts as neither a ply nor a game.
// kVirtual (a.node_v != nullptr, K = a.K > 1 leaves per step; never with kSolve): the warp runs descents
// j = 0 .. K-1 in order, descent j as simulation k + j on the virtual counts of the earlier ones, writes leaf row
// t*K + j, and adds its virtual visits along its path (lanes over the path) before the next descent.
template <bool kPuct, bool kSolve, bool kVirtual>
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_select_kernel(MctsArena a, int64_t count, uint64_t seed,
                                                                      uint32_t stream0, uint32_t k, double uct_c,
                                                                      uint32_t* __restrict__ leaf_dst,
                                                                      int32_t* __restrict__ out_status) {
  static_assert(!(kSolve && kVirtual), "the solver runs one leaf per step");
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  if constexpr (kVirtual) {
    select_descents<kPuct>(a, t, lane, seed, stream0 + static_cast<uint32_t>(t), k, uct_c, leaf_dst, out_status);
    return;
  }
  const int n = a.n, rw = a.rw;
  const uint32_t T = stream0 + static_cast<uint32_t>(t);
  int node = 0, depth = 0, nodes = a.tree[t].x;
  if constexpr (kSolve) {
    if (a.root_out[t] != 0) {
      if (leaf_dst == nullptr) {
        const uint4* root = reinterpret_cast<const uint4*>(a.node_rec + mcts_slot(a, t, 0) * rw);
        const uint4 hw = root[0];
        Header h;
        unpack_header(hw.x, hw.y, hw.z, hw.w, h);
        h.result = kDraw;
        uint4 o;
        pack_header(h, o.x, o.y, o.z, o.w);
        for (int r = 0; r < a.R; ++r) {
          uint4* dst = reinterpret_cast<uint4*>(a.roll_rec + (t * a.R + r) * rw);
          for (int q = lane; q < rw / 4; q += 32) dst[q] = q == 0 ? o : root[q];
        }
        for (int r = lane; r < a.R; r += 32)
          a.roll_ids[t * a.R + r] = mcts_rollout_stream(T, k, static_cast<uint32_t>(a.R), static_cast<uint32_t>(r));
      }
      if (lane == 0) {
        a.tree[t] = make_int4(nodes, 0, 0, kLeafSolved);
        if (out_status != nullptr) out_status[t] = kLeafSolved;
      }
      return;
    }
  }
  int2* path = a.path + t * a.P;
  bool terminal;
  for (;;) {
    const int64_t g = mcts_slot(a, t, node);
    uint32_t* rec = a.node_rec + g * rw;
    const uint4 hw = *reinterpret_cast<const uint4*>(rec);
    Header h;
    unpack_header(hw.x, hw.y, hw.z, hw.w, h);
    terminal = h.result != kOpen;
    const uint32_t visits = a.node_n[g];
    if (terminal || visits == 0u) break;
    const int64_t e0 = g * a.M;
    int legal = a.node_legal[g];
    int edge;
    if constexpr (kPuct) {
      // PUCT: the node was expanded at its first backup; warp argmax of (score, smaller key, lower edge)
      const double sq = mcts_sqrt_visits(visits);
      double best = 0.0;
      uint32_t bk = 0u;
      int bi = 0x7FFFFFFF;
      for (int i = lane; i < legal; i += 32) {
        const uint8_t o = a.edge_out[e0 + i];
        const double sc = o != 0 ? static_cast<double>(mcts_outcome_value(o))
                                 : mcts_puct_score(a.edge_w[e0 + i], a.edge_n[e0 + i], a.edge_p[e0 + i], sq, uct_c);
        const uint32_t key = a.edge_key[e0 + i];
        if (bi == 0x7FFFFFFF || mcts_puct_beats(sc, key, i, best, bk, bi)) {
          best = sc;
          bk = key;
          bi = i;
        }
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        const double os = __shfl_xor_sync(kFullMask, best, d);
        const uint32_t ok = __shfl_xor_sync(kFullMask, bk, d);
        const int oi = __shfl_xor_sync(kFullMask, bi, d);
        if (oi != 0x7FFFFFFF && (bi == 0x7FFFFFFF || mcts_puct_beats(os, ok, oi, best, bk, bi))) {
          best = os;
          bk = ok;
          bi = oi;
        }
      }
      edge = bi;
    } else {
      if (legal < 0) {
        legal = warp_expand(a, g, rec, h, lane);
        if constexpr (kSolve) {
          for (int i = lane; i < legal; i += 32) a.edge_out[e0 + i] = 0;
          __syncwarp();
        }
      }
      // unvisited edges
      int unvisited = 0;
      for (int i = lane; i < legal; i += 32) unvisited += a.edge_n[e0 + i] == 0u ? 1 : 0;
      unvisited = __reduce_add_sync(kFullMask, unvisited);
      if (unvisited > 0) {
        int j = static_cast<int>(mcts_draw(seed, T, k, static_cast<uint32_t>(unvisited)));
        edge = -1;
        for (int base = 0; edge < 0; base += 32) {
          const int i = base + lane;
          const uint32_t m = __ballot_sync(kFullMask, i < legal && a.edge_n[e0 + i] == 0u);
          const int c = __popc(m);
          if (j < c) edge = base + select_bit(m, j);
          else j -= c;
        }
      } else {
        const double log_parent = a.log_table[visits];
        double best = 0.0;
        int bi = 0x7FFFFFFF;
        for (int i = lane; i < legal; i += 32) {
          double s;
          if constexpr (kSolve) {
            // MCTS-Solver: a proven child scores its outcome (open_spiel uct_value)
            const uint8_t o = a.edge_out[e0 + i];
            s = o != 0 ? static_cast<double>(mcts_outcome_value(o))
                       : mcts_uct_score(a.edge_w[e0 + i], a.edge_n[e0 + i], log_parent, uct_c);
          } else {
            s = mcts_uct_score(a.edge_w[e0 + i], a.edge_n[e0 + i], log_parent, uct_c);
          }
          if (bi == 0x7FFFFFFF || mcts_score_beats(s, i, best, bi)) {
            best = s;
            bi = i;
          }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
          const double os = __shfl_xor_sync(kFullMask, best, d);
          const int oi = __shfl_xor_sync(kFullMask, bi, d);
          if (oi != 0x7FFFFFFF && (bi == 0x7FFFFFFF || mcts_score_beats(os, oi, best, bi))) {
            best = os;
            bi = oi;
          }
        }
        edge = bi;
      }
    }
    if (lane == 0) path[depth] = make_int2(node, (edge << 1) | static_cast<int>(h.ply & 1u));
    ++depth;
    int child = a.edge_child[e0 + edge];
    if (child < 0) {
      // the first visit of this edge: its child is the parent record with the move applied
      child = nodes++;
      const int64_t gc = mcts_slot(a, t, child);
      uint32_t* crec = a.node_rec + gc * rw;
      warp_copy_record(crec, rec, rw, lane);
      __syncwarp();
      if (lane == 0) {
        RecordRef<1> cb{crec, n};
        Header ch = h;
        const int action = a.edge_action[e0 + edge];
        const int x = action / n;
        apply_legal_cell<kMctsFloodStack>(cb, ch, x, action - x * n);
        uint4 o;
        pack_header(ch, o.x, o.y, o.z, o.w);
        *reinterpret_cast<uint4*>(crec) = o;
        a.node_legal[gc] = -1;
        a.node_n[gc] = 0u;
        a.edge_child[e0 + edge] = child;
        if ((kPuct || kSolve) && ch.result != kOpen)
          a.edge_out[e0 + edge] = mcts_outcome_code(ch, static_cast<int>(h.ply & 1u));
      }
      __syncwarp();
    }
    node = child;
  }
  const uint32_t* leaf = a.node_rec + mcts_slot(a, t, node) * rw;
  if (leaf_dst != nullptr) {
    warp_copy_record(leaf_dst + t * rw, leaf, rw, lane);
  } else {
    for (int r = 0; r < a.R; ++r) warp_copy_record(a.roll_rec + (t * a.R + r) * rw, leaf, rw, lane);
    for (int r = lane; r < a.R; r += 32)
      a.roll_ids[t * a.R + r] = mcts_rollout_stream(T, k, static_cast<uint32_t>(a.R), static_cast<uint32_t>(r));
  }
  const int status = terminal ? kLeafTerminal : kLeafNeedsValue;
  if (lane == 0) {
    a.tree[t] = make_int4(nodes, node, depth, status);
    if (out_status != nullptr) out_status[t] = status;
  }
}

// ---------------------------------------------------------------- backup ---
// kSolve: a finished tree's row is ignored, and a terminal leaf starts the MCTS-Solver proof pass up its path.
// kVirtual: rows j = 0 .. K-1 of the tree in order, each removing its virtual visits; a PUCT leaf is expanded by
// the lowest row whose leaf it is (later rows find it expanded and their priors are ignored).
template <bool kSolve, bool kVirtual>
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_backup_kernel(MctsArena a, int64_t count,
                                                                      const float* __restrict__ values,
                                                                      const float* __restrict__ priors,
                                                                      uint64_t seed, uint32_t stream0) {
  static_assert(!(kSolve && kVirtual), "the solver runs one leaf per step");
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int K = kVirtual ? a.K : 1;
  for (int j = 0; j < K; ++j) {  // K == 1 unless kVirtual
  const int64_t row = t * K + j;
  const int4 info = a.tree[row];
  if constexpr (kSolve) {
    if (info.w == kLeafSolved) return;
  }
  const int leaf = info.y, depth = info.z;
  double v[2];
  if (info.w == kLeafTerminal) {
    const uint4 hw = *reinterpret_cast<const uint4*>(a.node_rec + mcts_slot(a, t, leaf) * a.rw);
    Header h;
    unpack_header(hw.x, hw.y, hw.z, hw.w, h);
    mcts_terminal_value(h, v);
  } else if (values != nullptr) {
    v[0] = static_cast<double>(values[2 * row]);
    v[1] = static_cast<double>(values[2 * row + 1]);
  } else {
    // (double) sum_r ret_r[p] / R, r ascending
    double s0 = 0.0, s1 = 0.0;
    const float* ret = a.roll_ret + row * a.R * 2;
    for (int r = 0; r < a.R; ++r) {
      s0 = __dadd_rn(s0, static_cast<double>(ret[2 * r]));
      s1 = __dadd_rn(s1, static_cast<double>(ret[2 * r + 1]));
    }
    v[0] = __ddiv_rn(s0, static_cast<double>(a.R));
    v[1] = __ddiv_rn(s1, static_cast<double>(a.R));
  }
  const int2* path = a.path + row * a.P;
  for (int i = lane; i < depth; i += 32) {
    const int2 p = path[i];
    const int64_t g = mcts_slot(a, t, p.x);
    const int64_t e = g * a.M + (p.y >> 1);
    a.node_n[g] += 1u;
    a.edge_n[e] += 1u;
    a.edge_w[e] = __dadd_rn(a.edge_w[e], v[p.y & 1]);
    if constexpr (kVirtual) {
      a.node_v[g] -= 1;
      a.edge_v[e] -= 1;
    }
  }
  if (lane == 0) {
    a.node_n[mcts_slot(a, t, leaf)] += 1u;
    if constexpr (kVirtual) a.node_v[mcts_slot(a, t, leaf)] -= 1;
  }
  if (a.edge_p != nullptr && info.w != kLeafTerminal &&
      (!kVirtual || a.node_legal[mcts_slot(a, t, leaf)] < 0)) {
    // PUCT: expand the leaf with its priors (open_spiel expands on the second visit from evaluator.prior, which
    // AlphaZeroEvaluator answers from the network call that valued the leaf)
    const int64_t g = mcts_slot(a, t, leaf), e0 = g * a.M;
    const uint32_t* rec = a.node_rec + g * a.rw;
    const uint4 hw = *reinterpret_cast<const uint4*>(rec);
    Header h;
    unpack_header(hw.x, hw.y, hw.z, hw.w, h);
    const int legal = warp_expand(a, g, rec, h, lane);
    const float uniform = mcts_uniform_prior(legal);
    const float* prow = priors != nullptr ? priors + row * a.n * a.n : nullptr;
    const uint32_t T = stream0 + static_cast<uint32_t>(t);
    for (int i = lane; i < legal; i += 32) {
      a.edge_p[e0 + i] = prow != nullptr ? prow[a.edge_action[e0 + i]] : uniform;
      a.edge_key[e0 + i] = mcts_tie_key(seed, T, static_cast<uint32_t>(leaf), static_cast<uint32_t>(i));
      a.edge_out[e0 + i] = 0;
      if constexpr (kVirtual) a.edge_v[e0 + i] = 0;
    }
  }
  if constexpr (kVirtual) __syncwarp();  // the next row may update the same nodes and edges
  if constexpr (kSolve) {
    if (info.w == kLeafTerminal) {
      if (depth == 0) {
        // a terminal root is proven with its Returns()
        if (lane == 0) {
          const uint4 hw = *reinterpret_cast<const uint4*>(a.node_rec + mcts_slot(a, t, 0) * a.rw);
          Header h;
          unpack_header(hw.x, hw.y, hw.z, hw.w, h);
          a.root_out[t] = mcts_outcome_code(h, static_cast<int>(h.ply & 1u));
        }
        return;
      }
      // proof pass from the leaf's parent up: level i is path node i, whose edges' codes decide it; a proven node
      // writes its parent's edge (or the root code), which the next level reads
      for (int i = depth - 1; i >= 0; --i) {
        const int64_t g = mcts_slot(a, t, path[i].x), e0 = g * a.M;
        const int legal = a.node_legal[g];
        int mx = 0;
        bool all = true;
        for (int j = lane; j < legal; j += 32) {
          const int c = a.edge_out[e0 + j];
          mx = c > mx ? c : mx;
          all = all && c != 0;
        }
        mx = __reduce_max_sync(kFullMask, mx);
        all = __all_sync(kFullMask, all);
        const int pv = mcts_proven_value(mx, all);
        if (pv == kUnproven) break;
        if (lane == 0) {
          if (i > 0) {
            const int2 q = path[i - 1];
            a.edge_out[mcts_slot(a, t, q.x) * a.M + (q.y >> 1)] = mcts_parent_code(pv);
          } else {
            a.root_out[t] = static_cast<uint8_t>(2 + pv);
          }
        }
        __syncwarp();
      }
    }
  }
  }
}

// ------------------------------------------------------------ root stats ---
// BestChild of every search kind, open_spiel's sort_key (outcome value, N, W), then the tie key, then the lower edge:
// without outcome codes (UCT) every edge's outcome counts as 0, without tie keys (UCT, UCT solver) every key as 0.
// A PUCT root has no best move (-1) while no edge has a visit, a UCT root only while it has no edges, so that an
// expanded root queried between select and backup still reports edge 0.
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_root_stats_kernel(MctsArena a, int64_t count,
                                                                          int32_t* __restrict__ out_visits,
                                                                          double* __restrict__ out_value_sums,
                                                                          int32_t* __restrict__ out_best) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int cells = a.n * a.n;
  const int64_t g = mcts_slot(a, t, 0), e0 = g * a.M;
  const int legal = a.node_legal[g];
  for (int c = lane; c < cells; c += 32) {
    if (out_visits != nullptr) out_visits[t * cells + c] = 0;
    if (out_value_sums != nullptr) out_value_sums[t * cells + c] = 0.0;
  }
  __syncwarp();
  int bo = 0;
  uint32_t bn = 0u, bk = 0u, nmax = 0u;
  double bw = 0.0;
  int bi = 0x7FFFFFFF;
  for (int i = lane; i < legal; i += 32) {
    const int action = a.edge_action[e0 + i];
    const uint32_t en = a.edge_n[e0 + i];
    const double ew = a.edge_w[e0 + i];
    const int eo = a.edge_out != nullptr ? mcts_outcome_value(a.edge_out[e0 + i]) : 0;
    const uint32_t ek = a.edge_key != nullptr ? a.edge_key[e0 + i] : 0u;
    if (out_visits != nullptr) out_visits[t * cells + action] = static_cast<int32_t>(en);
    if (out_value_sums != nullptr) out_value_sums[t * cells + action] = ew;
    nmax = en > nmax ? en : nmax;
    if (bi == 0x7FFFFFFF || mcts_puct_best_beats(eo, en, ew, ek, i, bo, bn, bw, bk, bi)) {
      bo = eo;
      bn = en;
      bw = ew;
      bk = ek;
      bi = i;
    }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const int oo = __shfl_xor_sync(kFullMask, bo, d);
    const uint32_t on = __shfl_xor_sync(kFullMask, bn, d);
    const double ow = __shfl_xor_sync(kFullMask, bw, d);
    const uint32_t ok = __shfl_xor_sync(kFullMask, bk, d);
    const int oi = __shfl_xor_sync(kFullMask, bi, d);
    if (oi != 0x7FFFFFFF && (bi == 0x7FFFFFFF || mcts_puct_best_beats(oo, on, ow, ok, oi, bo, bn, bw, bk, bi))) {
      bo = oo;
      bn = on;
      bw = ow;
      bk = ok;
      bi = oi;
    }
  }
  nmax = __reduce_max_sync(kFullMask, nmax);
  const bool none = a.edge_p != nullptr ? nmax == 0u : legal <= 0;
  if (out_best != nullptr && lane == 0) out_best[t] = none ? -1 : static_cast<int32_t>(a.edge_action[e0 + bi]);
}

// ---------------------------------------------------------- solver stats ---
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_solver_stats_kernel(MctsArena a, int64_t count,
                                                                            uint8_t* __restrict__ out_proven,
                                                                            float* __restrict__ out_returns,
                                                                            int8_t* __restrict__ out_edge_values,
                                                                            int32_t* __restrict__ out_simulations) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int cells = a.n * a.n;
  const int64_t g = mcts_slot(a, t, 0), e0 = g * a.M;
  if (out_edge_values != nullptr) {
    for (int c = lane; c < cells; c += 32) out_edge_values[t * cells + c] = static_cast<int8_t>(kUnproven);
    __syncwarp();
    const int legal = a.node_legal[g];
    for (int i = lane; i < legal; i += 32) {
      const uint8_t o = a.edge_out[e0 + i];
      if (o != 0) out_edge_values[t * cells + a.edge_action[e0 + i]] = static_cast<int8_t>(mcts_outcome_value(o));
    }
  }
  if (lane == 0) {
    const uint8_t rc = a.root_out[t];
    if (out_proven != nullptr) out_proven[t] = rc != 0 ? 1 : 0;
    if (out_returns != nullptr) {
      // root.outcome: the code is for the root's player to move by ply parity
      const uint4 hw = *reinterpret_cast<const uint4*>(a.node_rec + g * a.rw);
      Header h;
      unpack_header(hw.x, hw.y, hw.z, hw.w, h);
      const int p = static_cast<int>(h.ply & 1u), v = mcts_outcome_value(rc);
      out_returns[2 * t + p] = static_cast<float>(v);
      out_returns[2 * t + 1 - p] = static_cast<float>(-v);
    }
    if (out_simulations != nullptr) out_simulations[t] = static_cast<int32_t>(a.node_n[g]);
  }
}

// --------------------------------------------------------------- advance ---
// Tree reuse (twixt_mcts_advance; semantics in twixt_mcts.cuh).  One warp per tree, three phases:
//   1. legality: the action's bit in the root's legal_word (lane = column); the root edge of the action by a
//      ballot over edge_action.  An edge without a child (or an unexpanded root) makes a fresh root: one lane
//      applies the move to slot 0's record, as select creates a child.
//   2. mark and rank, sequential in slot order from the new root s0: a slot is in the subtree when it is s0 or its
//      parent (a lower slot) kept it; kept slots get their rank in map[] until keep_nodes are ranked, the others
//      stay negative.  Lanes over a kept node's edges mark its children; a ballot over a window of 32 map entries
//      skips the slots that are not in the subtree.
//   3. move: each kept node, in ascending old slot order, goes to its rank r: the record with 16-byte stores and its
//      L edges' SoA entries (not M), children remapped through map[] and dropped children reset.
// The move is in place.  It is safe because r <= s - s0 <= s for every kept slot s, and slots are moved in
// ascending s: the destination r is either s itself (each lane rewrites the entries it has just read) or a lower
// slot, which is outside the subtree or was already moved.  So every source is read before its slot can be
// overwritten.  map[] is per-tree scratch, not part of the tree.  The V counts (K > 1) are 0 between steps and are
// written as 0 at the destinations.
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_advance_kernel(MctsArena a, int64_t count,
                                                                       const int32_t* __restrict__ actions,
                                                                       int keep_nodes, int32_t* map_all,
                                                                       int32_t* __restrict__ out_status,
                                                                       unsigned int* __restrict__ illegal_index) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int n = a.n, rw = a.rw, M = a.M;
  int4* entry = a.tree + t * a.K;
  const int nodes = entry->x;
  const int action = actions[t];
  const int64_t root = mcts_slot(a, t, 0), r0 = root * M;
  uint32_t* rrec = a.node_rec + root * rw;
  const uint4 hw = *reinterpret_cast<const uint4*>(rrec);
  Header h;
  unpack_header(hw.x, hw.y, hw.z, hw.w, h);

  // 1. legality and the root edge
  int s0 = 0;        // old slot of the new root, -1: a fresh root
  uint8_t code = 0;  // outcome code of the chosen edge
  if (action != -1) {
    bool legal = false;
    if (h.result == kOpen && action >= 0 && action < n * n) {
      RecordRef<1> b{rrec, n};
      const int x = action / n;
      const uint32_t w = lane < n ? legal_word(b, h, lane) : 0u;
      legal = ((__shfl_sync(kFullMask, w, x) >> (action - x * n)) & 1u) != 0u;
    }
    if (!legal) {
      if (lane == 0) {
        if (out_status != nullptr) out_status[t] = kRootIllegal;
        atomicMin(illegal_index, static_cast<unsigned int>(t));  // the host names this action in its message
      }
      return;
    }
    s0 = -1;
    const int L = a.node_legal[root];
    for (int base = 0; base < L; base += 32) {
      const int i = base + lane;
      const unsigned m = __ballot_sync(kFullMask, i < L && a.edge_action[r0 + i] == action);
      if (m != 0u) {
        const int e = base + __ffs(static_cast<int>(m)) - 1;
        s0 = a.edge_child[r0 + e];
        if (a.edge_out != nullptr) code = a.edge_out[r0 + e];
        break;
      }
    }
    if (s0 < 0) {
      // no child: the root with the move applied, cleared as begin clears a tree
      if (lane == 0) {
        RecordRef<1> b{rrec, n};
        const int x = action / n;
        apply_legal_cell<kMctsFloodStack>(b, h, x, action - x * n);
        uint4 o;
        pack_header(h, o.x, o.y, o.z, o.w);
        *reinterpret_cast<uint4*>(rrec) = o;
        a.node_legal[root] = -1;
        a.node_n[root] = 0u;
        if (a.node_v != nullptr) a.node_v[root] = 0;
        if (a.root_out != nullptr) a.root_out[t] = mcts_advanced_root_code(code);
        entry->x = 1;
        if (out_status != nullptr) out_status[t] = kRootFresh;
      }
      return;
    }
  }

  // 2. mark and rank: map = -1 outside the subtree, -2 marked (a kept parent's child), >= 0 the rank
  int32_t* map = map_all + t * a.S;
  for (int s = s0 + 1 + lane; s < nodes; s += 32) map[s] = -1;
  if (lane == 0) map[s0] = -2;
  __syncwarp();
  int kept = 0;
  for (int s = s0; s < nodes && kept < keep_nodes;) {
    const int q = s + lane;
    const unsigned m = __ballot_sync(kFullMask, q < nodes && map[q] != -1);
    if (m == 0u) {
      s += 32;
      continue;
    }
    s += __ffs(static_cast<int>(m)) - 1;  // the next slot in the subtree
    const int64_t g = mcts_slot(a, t, s), e0 = g * M;
    const int L = a.node_legal[g];
    for (int i = lane; i < L; i += 32) {
      const int c = a.edge_child[e0 + i];
      if (c >= 0) map[c] = -2;
    }
    if (lane == 0) map[s] = kept;
    ++kept;
    ++s;
    __syncwarp();
  }

  // 3. move the kept nodes down to their ranks
  uint32_t root_visits = 0u;
  for (int s = s0, moved = 0; moved < kept;) {
    const int q = s + lane;
    const unsigned m = __ballot_sync(kFullMask, q < nodes && map[q] >= 0);
    if (m == 0u) {
      s += 32;
      continue;
    }
    s += __ffs(static_cast<int>(m)) - 1;
    const int r = moved++;
    const int64_t gs = mcts_slot(a, t, s), gr = mcts_slot(a, t, r), es = gs * M, er = gr * M;
    const int L = a.node_legal[gs];
    const uint32_t visits = a.node_n[gs];
    if (r == 0) root_visits = visits;
    if (r != s) warp_copy_record(a.node_rec + gr * rw, a.node_rec + gs * rw, rw, lane);
    for (int i = lane; i < L; i += 32) {
      const int c = a.edge_child[es + i];
      const int mc = c >= 0 ? map[c] : -1;
      const bool dropped = c >= 0 && mc < 0;  // cut by keep_nodes: unvisited again
      const uint32_t en = dropped ? 0u : a.edge_n[es + i];
      const double ew = dropped ? 0.0 : a.edge_w[es + i];
      if (r != s) {
        a.edge_action[er + i] = a.edge_action[es + i];
        if (a.edge_p != nullptr) {
          a.edge_p[er + i] = a.edge_p[es + i];
          a.edge_key[er + i] = a.edge_key[es + i];
        }
        if (a.edge_out != nullptr) a.edge_out[er + i] = a.edge_out[es + i];
      }
      a.edge_n[er + i] = en;
      a.edge_w[er + i] = ew;
      a.edge_child[er + i] = c >= 0 ? (mc >= 0 ? mc : -1) : -1;
      if (a.edge_v != nullptr) a.edge_v[er + i] = 0;
    }
    __syncwarp();  // every lane has read slot s before lane 0 writes slot r
    if (lane == 0) {
      a.node_legal[gr] = L;
      a.node_n[gr] = visits;
      if (a.node_v != nullptr) a.node_v[gr] = 0;
    }
    ++s;
  }
  if (lane == 0) {
    entry->x = kept;
    if (action != -1 && a.root_out != nullptr) a.root_out[t] = mcts_advanced_root_code(code);
    if (out_status != nullptr) out_status[t] = root_visits > 0u ? kRootKept : kRootFresh;
  }
}

// ------------------------------------------------------ set root priors ---
// P(a) of every root edge of each expanded root from priors [count, n*n]; unexpanded roots are left alone
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_set_root_priors_kernel(MctsArena a, int64_t count,
                                                                               const float* __restrict__ priors) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int64_t g = mcts_slot(a, t, 0), e0 = g * a.M;
  const int legal = a.node_legal[g];
  const float* row = priors + t * a.n * a.n;
  for (int i = lane; i < legal; i += 32) a.edge_p[e0 + i] = row[a.edge_action[e0 + i]];
}

// ------------------------------------------------------ Gumbel AlphaZero ---
// Semantics in twixt_mcts.cuh.  Every reduction over a node's edges is lanes over the edges (lane l takes edges l,
// l+32, .. in ascending order), then an xor butterfly, so that a sum has the order of mcts_lane_sums in every lane.
__device__ __forceinline__ double warp_sum(double s) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) s = __dadd_rn(s, __shfl_xor_sync(kFullMask, s, d));
  return s;
}
__device__ __forceinline__ double warp_max(double x) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) x = mcts_max(x, __shfl_xor_sync(kFullMask, x, d));
  return x;
}
__device__ __forceinline__ double warp_min(double x) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) x = mcts_min(x, __shfl_xor_sync(kFullMask, x, d));
  return x;
}
// (score, edge) argmax over the lanes: the larger score, then the lower edge; bi = 0x7FFFFFFF for none
__device__ __forceinline__ int warp_argmax(double best, int bi) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const double os = __shfl_xor_sync(kFullMask, best, d);
    const int oi = __shfl_xor_sync(kFullMask, bi, d);
    if (oi != 0x7FFFFFFF && (bi == 0x7FFFFFFF || mcts_score_beats(os, oi, best, bi))) {
      best = os;
      bi = oi;
    }
  }
  return bi;
}

// What sigma(a) of a node's edges needs: max l, SN, max N, v_mix and the min / max / scale of q^
struct GumbelNode {
  double max_logit, v_mix, q_min, q_max, scale;
  uint32_t sum_n, max_n;
};

// The completed-Q transform of the expanded node at global slot g with L = legal edges (every lane gets the same)
__device__ GumbelNode gumbel_node(const MctsArena& a, const MctsGumbel& gm, int64_t g, int legal, int lane) {
  const int64_t e0 = g * a.M;
  GumbelNode s;
  double mx = -INFINITY;
  uint32_t sn = 0u, mn = 0u;
  for (int i = lane; i < legal; i += 32) {
    mx = mcts_max(mx, static_cast<double>(gm.edge_logit[e0 + i]));
    const uint32_t n = a.edge_n[e0 + i];
    sn += n;
    mn = n > mn ? n : mn;
  }
  s.max_logit = warp_max(mx);
  s.sum_n = __reduce_add_sync(kFullMask, sn);
  s.max_n = __reduce_max_sync(kFullMask, mn);
  double weighted_q = 0.0;
  if (s.sum_n > 0u) {  // with no visited edge both sums below are 0.0
    double z = 0.0;
    for (int i = lane; i < legal; i += 32)
      z = __dadd_rn(z, mcts_exp(__dsub_rn(static_cast<double>(gm.edge_logit[e0 + i]), s.max_logit)));
    z = warp_sum(z);
    double sp = 0.0;
    for (int i = lane; i < legal; i += 32)
      if (a.edge_n[e0 + i] > 0u)
        sp = __dadd_rn(sp, mcts_gumbel_prob(mcts_exp(__dsub_rn(static_cast<double>(gm.edge_logit[e0 + i]),
                                                               s.max_logit)), z));
    sp = warp_sum(sp);
    for (int i = lane; i < legal; i += 32) {
      const uint32_t n = a.edge_n[e0 + i];
      if (n > 0u) {
        const double pi = mcts_gumbel_prob(mcts_exp(__dsub_rn(static_cast<double>(gm.edge_logit[e0 + i]), s.max_logit)), z);
        weighted_q = __dadd_rn(weighted_q, mcts_gumbel_mix_term(pi, a.edge_w[e0 + i], n, sp));
      }
    }
    weighted_q = warp_sum(weighted_q);
  }
  s.v_mix = mcts_gumbel_mixed_value(gm.node_value[g], s.sum_n, weighted_q);
  double qmin = INFINITY, qmax = -INFINITY;
  for (int i = lane; i < legal; i += 32) {
    const double q = mcts_gumbel_completed_q(a.edge_w[e0 + i], a.edge_n[e0 + i], s.v_mix);
    qmin = mcts_min(qmin, q);
    qmax = mcts_max(qmax, q);
  }
  s.q_min = warp_min(qmin);
  s.q_max = warp_max(qmax);
  s.scale = mcts_gumbel_scale(gm.c_visit, gm.c_scale, s.max_n);
  return s;
}

// sigma(a) of edge e
__device__ __forceinline__ double gumbel_sigma(const MctsArena& a, const GumbelNode& s, int64_t e) {
  const double q = mcts_gumbel_completed_q(a.edge_w[e], a.edge_n[e], s.v_mix);
  return mcts_gumbel_sigma(q, s.q_min, s.q_max, s.scale);
}

// l(a) + sigma(a) of edge e
__device__ __forceinline__ double gumbel_completed_logit(const MctsGumbel& gm, const MctsArena& a, const GumbelNode& s,
                                                         int64_t e) {
  return __dadd_rn(static_cast<double>(gm.edge_logit[e]), gumbel_sigma(a, s, e));
}

// max over the edges of l + sigma and the sum of mcts_exp(l + sigma - that max): softmax(l + sigma) = e / z
__device__ __forceinline__ void gumbel_softmax_norm(const MctsArena& a, const MctsGumbel& gm, const GumbelNode& s,
                                                    int64_t e0, int legal, int lane, double& mx, double& z) {
  double m = -INFINITY;
  for (int i = lane; i < legal; i += 32) m = mcts_max(m, gumbel_completed_logit(gm, a, s, e0 + i));
  mx = warp_max(m);
  double sum = 0.0;
  for (int i = lane; i < legal; i += 32)
    sum = __dadd_rn(sum, mcts_exp(__dsub_rn(gumbel_completed_logit(gm, a, s, e0 + i), mx)));
  z = warp_sum(sum);
}

// the root's edge among those with N(a) = considered (-1: none eligible, the lowest edge), by the root score
__device__ __forceinline__ int gumbel_root_argmax(const MctsArena& a, const MctsGumbel& gm, const GumbelNode& s,
                                                  int64_t t, int64_t e0, int legal, int64_t considered, int lane) {
  const float* noise = gm.root_gumbel + t * a.n * a.n;
  double best = 0.0;
  int bi = 0x7FFFFFFF;
  for (int i = lane; i < legal; i += 32) {
    if (static_cast<int64_t>(a.edge_n[e0 + i]) != considered) continue;
    const double sc = mcts_gumbel_root_score(noise[a.edge_action[e0 + i]], gm.edge_logit[e0 + i], s.max_logit,
                                             gumbel_sigma(a, s, e0 + i));
    if (bi == 0x7FFFFFFF || mcts_score_beats(sc, i, best, bi)) {
      best = sc;
      bi = i;
    }
  }
  bi = warp_argmax(best, bi);
  return bi == 0x7FFFFFFF ? 0 : bi;
}

// ------------------------------------------------------------------ Gumbel select ---
// One warp per tree, one descent (K = 1, no solver): the root takes Sequential Halving's edge, every other node the
// interior rule; a chosen edge without a child creates it as the PUCT select does.  The leaf goes to leaf_dst + t*rw
// or to the R rollout slots, as mcts_select_kernel writes it.
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_gumbel_select_kernel(MctsArena a, MctsGumbel gm, int64_t count,
                                                                             uint32_t stream0, uint32_t k,
                                                                             uint32_t* __restrict__ leaf_dst,
                                                                             int32_t* __restrict__ out_status) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int n = a.n, rw = a.rw;
  const uint32_t T = stream0 + static_cast<uint32_t>(t);
  int node = 0, depth = 0, nodes = a.tree[t].x;
  int2* path = a.path + t * a.P;
  bool terminal;
  for (;;) {
    const int64_t g = mcts_slot(a, t, node);
    uint32_t* rec = a.node_rec + g * rw;
    const uint4 hw = *reinterpret_cast<const uint4*>(rec);
    Header h;
    unpack_header(hw.x, hw.y, hw.z, hw.w, h);
    terminal = h.result != kOpen;
    if (terminal || a.node_n[g] == 0u) break;
    const int64_t e0 = g * a.M;
    const int legal = a.node_legal[g];
    const GumbelNode s = gumbel_node(a, gm, g, legal, lane);
    int edge;
    if (node == 0) {
      const int m = gm.max_considered < legal ? gm.max_considered : legal;
      const int64_t considered =
          static_cast<int>(s.sum_n) < gm.cols ? gm.table[static_cast<int64_t>(m) * gm.cols + s.sum_n] : -1;
      edge = gumbel_root_argmax(a, gm, s, t, e0, legal, considered, lane);
    } else {
      double mx, z;
      gumbel_softmax_norm(a, gm, s, e0, legal, lane, mx, z);
      double best = 0.0;
      int bi = 0x7FFFFFFF;
      for (int i = lane; i < legal; i += 32) {
        const double e = mcts_exp(__dsub_rn(gumbel_completed_logit(gm, a, s, e0 + i), mx));
        const double sc = mcts_gumbel_interior_score(e, z, a.edge_n[e0 + i], s.sum_n);
        if (bi == 0x7FFFFFFF || mcts_score_beats(sc, i, best, bi)) {
          best = sc;
          bi = i;
        }
      }
      edge = warp_argmax(best, bi);
    }
    if (lane == 0) path[depth] = make_int2(node, (edge << 1) | static_cast<int>(h.ply & 1u));
    ++depth;
    int child = a.edge_child[e0 + edge];
    if (child < 0) {
      child = nodes++;
      const int64_t gc = mcts_slot(a, t, child);
      uint32_t* crec = a.node_rec + gc * rw;
      warp_copy_record(crec, rec, rw, lane);
      __syncwarp();
      if (lane == 0) {
        RecordRef<1> cb{crec, n};
        Header ch = h;
        const int action = a.edge_action[e0 + edge];
        const int x = action / n;
        apply_legal_cell<kMctsFloodStack>(cb, ch, x, action - x * n);
        uint4 o;
        pack_header(ch, o.x, o.y, o.z, o.w);
        *reinterpret_cast<uint4*>(crec) = o;
        a.node_legal[gc] = -1;
        a.node_n[gc] = 0u;
        a.edge_child[e0 + edge] = child;
      }
      __syncwarp();
    }
    node = child;
  }
  const uint32_t* leaf = a.node_rec + mcts_slot(a, t, node) * rw;
  if (leaf_dst != nullptr) {
    warp_copy_record(leaf_dst + t * rw, leaf, rw, lane);
  } else {
    for (int r = 0; r < a.R; ++r) warp_copy_record(a.roll_rec + (t * a.R + r) * rw, leaf, rw, lane);
    for (int r = lane; r < a.R; r += 32)
      a.roll_ids[t * a.R + r] = mcts_rollout_stream(T, k, static_cast<uint32_t>(a.R), static_cast<uint32_t>(r));
  }
  const int status = terminal ? kLeafTerminal : kLeafNeedsValue;
  if (lane == 0) {
    a.tree[t] = make_int4(nodes, node, depth, status);
    if (out_status != nullptr) out_status[t] = status;
  }
}

// ------------------------------------------------------------------ Gumbel backup ---
// The leaf value as mcts_backup_kernel takes it, added along the path; the leaf's raw value v(leaf) is that value for
// its player to move, and a non-terminal leaf is expanded with l(a) = logits[t, action] (0 without logits).
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_gumbel_backup_kernel(MctsArena a, MctsGumbel gm, int64_t count,
                                                                             const float* __restrict__ values,
                                                                             const float* __restrict__ logits) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int4 info = a.tree[t];
  const int leaf = info.y, depth = info.z;
  const int64_t gl = mcts_slot(a, t, leaf);
  const uint32_t* rec = a.node_rec + gl * a.rw;
  const uint4 hw = *reinterpret_cast<const uint4*>(rec);
  Header h;
  unpack_header(hw.x, hw.y, hw.z, hw.w, h);
  double v[2];
  if (info.w == kLeafTerminal) {
    mcts_terminal_value(h, v);
  } else if (values != nullptr) {
    v[0] = static_cast<double>(values[2 * t]);
    v[1] = static_cast<double>(values[2 * t + 1]);
  } else {
    double s0 = 0.0, s1 = 0.0;
    const float* ret = a.roll_ret + t * a.R * 2;
    for (int r = 0; r < a.R; ++r) {
      s0 = __dadd_rn(s0, static_cast<double>(ret[2 * r]));
      s1 = __dadd_rn(s1, static_cast<double>(ret[2 * r + 1]));
    }
    v[0] = __ddiv_rn(s0, static_cast<double>(a.R));
    v[1] = __ddiv_rn(s1, static_cast<double>(a.R));
  }
  const int2* path = a.path + t * a.P;
  for (int i = lane; i < depth; i += 32) {
    const int2 p = path[i];
    const int64_t g = mcts_slot(a, t, p.x);
    const int64_t e = g * a.M + (p.y >> 1);
    a.node_n[g] += 1u;
    a.edge_n[e] += 1u;
    a.edge_w[e] = __dadd_rn(a.edge_w[e], v[p.y & 1]);
  }
  if (lane == 0) {
    a.node_n[gl] += 1u;
    gm.node_value[gl] = (h.ply & 1u) != 0u ? v[1] : v[0];
  }
  if (info.w != kLeafTerminal) {
    const int64_t e0 = gl * a.M;
    const int legal = warp_expand(a, gl, rec, h, lane);
    const float* row = logits != nullptr ? logits + t * a.n * a.n : nullptr;
    for (int i = lane; i < legal; i += 32) gm.edge_logit[e0 + i] = row != nullptr ? row[a.edge_action[e0 + i]] : 0.0f;
  }
}

// -------------------------------------------------------------- set root gumbel ---
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_set_root_gumbel_kernel(MctsArena a, MctsGumbel gm, int64_t count,
                                                                               const float* __restrict__ gumbel) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int cells = a.n * a.n;
  for (int c = lane; c < cells; c += 32) gm.root_gumbel[t * cells + c] = gumbel[t * cells + c];
}

// ------------------------------------------------------------------ Gumbel stats ---
// The action (the root score among the edges of most visits; -1 for a terminal or unexpanded root) and the improved
// policy softmax(l + sigma) at the root's action cells (0 elsewhere, all 0 for a terminal or unexpanded root)
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_gumbel_stats_kernel(MctsArena a, MctsGumbel gm, int64_t count,
                                                                            int32_t* __restrict__ out_action,
                                                                            float* __restrict__ out_policy) {
  const int lane = threadIdx.x & 31;
  const int64_t t = blockIdx.x * static_cast<int64_t>(kMctsWarps) + (threadIdx.x >> 5);
  if (t >= count) return;
  const int cells = a.n * a.n;
  const int64_t g = mcts_slot(a, t, 0), e0 = g * a.M;
  const int legal = a.node_legal[g];
  if (out_policy != nullptr) {
    for (int c = lane; c < cells; c += 32) out_policy[t * cells + c] = 0.0f;
    __syncwarp();
  }
  if (legal < 0) {
    if (out_action != nullptr && lane == 0) out_action[t] = -1;
    return;
  }
  const GumbelNode s = gumbel_node(a, gm, g, legal, lane);
  if (out_action != nullptr) {
    const int edge = gumbel_root_argmax(a, gm, s, t, e0, legal, s.max_n, lane);
    if (lane == 0) out_action[t] = a.edge_action[e0 + edge];
  }
  if (out_policy != nullptr) {
    double mx, z;
    gumbel_softmax_norm(a, gm, s, e0, legal, lane, mx, z);
    for (int i = lane; i < legal; i += 32)
      out_policy[t * cells + a.edge_action[e0 + i]] =
          __double2float_rn(__ddiv_rn(mcts_exp(__dsub_rn(gumbel_completed_logit(gm, a, s, e0 + i), mx)), z));
  }
}

// One warp per tree: count trees in blocks of kMctsWarps warps, nothing to launch for none
template <typename... Params, typename... Args>
cudaError_t launch_per_tree(void (*kernel)(Params...), int64_t count, cudaStream_t s, Args... args) {
  if (count <= 0) return cudaSuccess;
  kernel<<<static_cast<unsigned>((count + kMctsWarps - 1) / kMctsWarps), kMctsWarps * 32, 0, s>>>(args...);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_mcts_begin(const MctsArena& a, const uint32_t* roots, int64_t count, cudaStream_t s) {
  return launch_per_tree(mcts_begin_kernel, count, s, a, roots, count);
}

cudaError_t launch_mcts_select(const MctsArena& a, int64_t count, uint64_t seed, uint32_t stream0, uint32_t k,
                               double uct_c, uint32_t* leaf_dst, int32_t* out_status, cudaStream_t s) {
  const bool puct = a.edge_p != nullptr, solve = a.root_out != nullptr;
  auto kernel = a.node_v != nullptr
                    ? (puct ? mcts_select_kernel<true, false, true> : mcts_select_kernel<false, false, true>)
                : puct ? (solve ? mcts_select_kernel<true, true, false> : mcts_select_kernel<true, false, false>)
                       : (solve ? mcts_select_kernel<false, true, false> : mcts_select_kernel<false, false, false>);
  return launch_per_tree(kernel, count, s, a, count, seed, stream0, k, uct_c, leaf_dst, out_status);
}

cudaError_t launch_mcts_backup(const MctsArena& a, int64_t count, const float* values, const float* priors,
                               uint64_t seed, uint32_t stream0, cudaStream_t s) {
  auto kernel = a.node_v != nullptr ? mcts_backup_kernel<false, true>
                                    : (a.root_out != nullptr ? mcts_backup_kernel<true, false>
                                                             : mcts_backup_kernel<false, false>);
  return launch_per_tree(kernel, count, s, a, count, values, priors, seed, stream0);
}

cudaError_t launch_mcts_root_stats(const MctsArena& a, int64_t count, int32_t* out_visits, double* out_value_sums,
                                   int32_t* out_best, cudaStream_t s) {
  return launch_per_tree(mcts_root_stats_kernel, count, s, a, count, out_visits, out_value_sums, out_best);
}

cudaError_t launch_mcts_solver_stats(const MctsArena& a, int64_t count, uint8_t* out_proven, float* out_returns,
                                     int8_t* out_edge_values, int32_t* out_simulations, cudaStream_t s) {
  return launch_per_tree(mcts_solver_stats_kernel, count, s, a, count, out_proven, out_returns, out_edge_values,
                         out_simulations);
}

cudaError_t launch_mcts_advance(const MctsArena& a, int64_t count, const int32_t* actions, int keep_nodes,
                                int32_t* map, int32_t* out_status, unsigned int* illegal_index, cudaStream_t s) {
  return launch_per_tree(mcts_advance_kernel, count, s, a, count, actions, keep_nodes, map, out_status,
                         illegal_index);
}

cudaError_t launch_mcts_set_root_priors(const MctsArena& a, int64_t count, const float* priors, cudaStream_t s) {
  return launch_per_tree(mcts_set_root_priors_kernel, count, s, a, count, priors);
}

cudaError_t launch_mcts_gumbel_select(const MctsArena& a, const MctsGumbel& gm, int64_t count, uint32_t stream0,
                                      uint32_t k, uint32_t* leaf_dst, int32_t* out_status, cudaStream_t s) {
  return launch_per_tree(mcts_gumbel_select_kernel, count, s, a, gm, count, stream0, k, leaf_dst, out_status);
}

cudaError_t launch_mcts_gumbel_backup(const MctsArena& a, const MctsGumbel& gm, int64_t count, const float* values,
                                      const float* logits, cudaStream_t s) {
  return launch_per_tree(mcts_gumbel_backup_kernel, count, s, a, gm, count, values, logits);
}

cudaError_t launch_mcts_set_root_gumbel(const MctsArena& a, const MctsGumbel& gm, int64_t count, const float* gumbel,
                                        cudaStream_t s) {
  return launch_per_tree(mcts_set_root_gumbel_kernel, count, s, a, gm, count, gumbel);
}

cudaError_t launch_mcts_gumbel_stats(const MctsArena& a, const MctsGumbel& gm, int64_t count, int32_t* out_action,
                                     float* out_policy, cudaStream_t s) {
  return launch_per_tree(mcts_gumbel_stats_kernel, count, s, a, gm, count, out_action, out_policy);
}

}  // namespace twixt
