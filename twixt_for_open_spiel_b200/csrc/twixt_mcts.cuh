// twixt_mcts.cuh -- the scalar pieces of the batched MCTS search (twixt_mcts.cu), shared with the host
// harness tests/mcts_harness.cc so that the search arithmetic can be checked without a GPU.
//
// Search semantics (open_spiel MCTSBot with RandomRolloutEvaluator, solve = false, no Dirichlet noise, made
// deterministic): see include/twixt_b200.h, "Batched MCTS".  Everything that decides which edge a simulation
// takes lives here:
//   uct score            q = W/N, e = c * sqrt(L[N(s)] / N), score = q + e in IEEE double, no contraction
//   unvisited-edge draw  word 0 of Philox4x32-10(key = seed, counter = (T lo, T hi, k, 1)), index (w*U) >> 32
//   rollout stream id    (T << 32) | (k*R + r)
//   best child           most visits, then larger W, then lowest action
//
// Storage of one tree (S = max_simulations + 1 node slots, M = max_legal_actions = n(n-2),
// rw = record_words(n), P = min(max_simulations, max_game_length) + 1 path entries, R = n_rollouts):
//   per node   rw*4 (record) + 4 (legal count, -1 = not expanded) + 4 (visit count N(s))
//              + M * (2 + 4 + 8 + 4) (edges, SoA: action u16, N u32, W f64, child i32)
//   per tree   16 (node count, leaf slot, path length, leaf status) + P*8 (path)
//              + R * (rw*4 + 8 + 8) (rollout slot records, stream ids, float returns)
//   bytes per tree = S * (rw*4 + 8 + 18*M) + 16 + 8*P + R * (rw*4 + 16)
// plus one table of (max_simulations + 1) doubles per search.  At n = 12 a node is 2 616 bytes.
#pragma once
#include <stdint.h>

#include "twixt_engine.cuh"
#include "twixt_philox.cuh"

#if !defined(__CUDA_ARCH__)
#include <cmath>
#endif

namespace twixt {

enum : int { kLeafNeedsValue = 0, kLeafTerminal = 1 };

struct MctsSizes {
  int64_t slots;      // node slots per tree (max_simulations + 1)
  int64_t edges;      // edges per node (max_legal_actions)
  int64_t path;       // path entries per tree
  int64_t rw;         // record words
  int64_t rollouts;   // R
};

TW_HD MctsSizes mcts_sizes(int n, int max_simulations, int n_rollouts) {
  MctsSizes s;
  const int max_game_length = n * n - 4 + 1;
  s.slots = static_cast<int64_t>(max_simulations) + 1;
  s.edges = static_cast<int64_t>(n) * (n - 2);
  s.path = static_cast<int64_t>(max_simulations < max_game_length ? max_simulations : max_game_length) + 1;
  s.rw = record_words(n);
  s.rollouts = n_rollouts;
  return s;
}

// the formula of the header comment above
TW_HD int64_t mcts_bytes_per_tree(const MctsSizes& s) {
  return s.slots * (s.rw * 4 + 8 + 18 * s.edges) + 16 + 8 * s.path + s.rollouts * (s.rw * 4 + 16);
}

// UCT score of an edge with N(a) = n > 0 visits and value sum w, under a parent whose ln N(s) is log_parent.
// Bit-identical on the device and on a host compiled with -ffp-contract=off.
TW_HD double mcts_uct_score(double w, uint32_t n, double log_parent, double c) {
  const double nd = static_cast<double>(n);
#if defined(__CUDA_ARCH__)
  const double q = __ddiv_rn(w, nd);
  const double e = __dmul_rn(c, __dsqrt_rn(__ddiv_rn(log_parent, nd)));
  return __dadd_rn(q, e);
#else
  const double q = w / nd;
  const double e = c * std::sqrt(log_parent / nd);
  return q + e;
#endif
}

// (score a, edge ia) beats (score b, edge ib): the larger score, then the lower edge (= lower action)
TW_HD bool mcts_score_beats(double a, int ia, double b, int ib) { return a > b || (a == b && ia < ib); }

// BestChild: (visits, value sum, edge) beats another: most visits, then larger W, then the lower action
TW_HD bool mcts_best_beats(uint32_t na, double wa, int ia, uint32_t nb, double wb, int ib) {
  if (na != nb) return na > nb;
  if (wa != wb) return wa > wb;
  return ia < ib;
}

// the one random draw of simulation k of the tree with stream id T: the index of the unvisited edge taken,
// among U >= 1 unvisited edges in ascending action order
TW_HD uint32_t mcts_draw(uint64_t seed, uint32_t tree_stream, uint32_t k, uint32_t unvisited) {
  uint32_t r[4];
  philox4x32_10(tree_stream, 0u, k, 1u, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), r);
  return playout_index(r[0], unvisited);
}

// Philox stream of rollout r of simulation k (R rollouts per simulation)
TW_HD uint64_t mcts_rollout_stream(uint32_t tree_stream, uint32_t k, uint32_t R, uint32_t r) {
  return (static_cast<uint64_t>(tree_stream) << 32) | static_cast<uint64_t>(k * R + r);
}

// Returns() of a terminal header (twixt.h:50-63), as the doubles a backup adds
TW_HD void mcts_terminal_value(const Header& h, double v[2]) {
  v[0] = h.result == kRedWin ? 1.0 : (h.result == kBlueWin ? -1.0 : 0.0);
  v[1] = h.result == kBlueWin ? 1.0 : (h.result == kRedWin ? -1.0 : 0.0);
}

}  // namespace twixt
