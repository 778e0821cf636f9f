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
// and, for a PUCT search (twixt_mcts_create_puct):
//   puct score           q = N(a) > 0 ? W/N(a) : 0, u = ((c * P) * sqrt(N(s))) / (N(a) + 1), q + u in IEEE
//                        double, no contraction; an edge whose child is terminal scores Returns()[player at s]
//   tie key              word 0 of Philox4x32-10(key = seed, counter = (T, node slot, edge, 2)); among equal
//                        scores the smaller key wins, then the lower edge
//   best child           (terminal outcome or 0, N, W), then the tie key, then the lower edge
//
// Storage of one tree (S = max_simulations + 1 node slots, M = max_legal_actions = n(n-2),
// rw = record_words(n), P = min(max_simulations, max_game_length) + 1 path entries, R = n_rollouts):
//   per node   rw*4 (record) + 4 (legal count, -1 = not expanded) + 4 (visit count N(s))
//              + M * (2 + 4 + 8 + 4) (edges, SoA: action u16, N u32, W f64, child i32)
//   per tree   16 (node count, leaf slot, path length, leaf status) + P*8 (path)
//              + R * (rw*4 + 8 + 8) (rollout slot records, stream ids, float returns)
//   bytes per tree = S * (rw*4 + 8 + 18*M) + 16 + 8*P + R * (rw*4 + 16)
// plus one table of (max_simulations + 1) doubles per search.  At n = 12 a node is 2 616 bytes.
// A PUCT search adds per edge 4 (prior P f32) + 4 (tie key u32) + 1 (terminal outcome u8):
//   PUCT bytes per tree = S * (rw*4 + 8 + 27*M) + 16 + 8*P + R * (rw*4 + 16)
// A solver search (TWIXT_MCTS_SOLVE, MCTS-Solver) adds 1 per tree (root outcome code u8); a UCT one also the
// outcome byte per edge, which PUCT already has:
//   UCT + solve bytes per tree  = S * (rw*4 + 8 + 19*M) + 17 + 8*P + R * (rw*4 + 16)
//   PUCT + solve bytes per tree = S * (rw*4 + 8 + 27*M) + 17 + 8*P + R * (rw*4 + 16)
// The outcome code of an edge is 0 while its child is unproven, else 2 + the child's value for the player to move
// at the parent (1 = loss, 2 = draw, 3 = win); the root code is 2 + the root's value for its own player to move
// (ply parity, also for a terminal root).
//
// Several leaves per step (twixt_mcts_create_parallel, K = leaves_per_step > 1, virtual loss vl): one step is K
// descents j = 0 .. K-1 of every tree, descent j being simulation k = sims_since_begin + j (draw and rollout
// streams as above).  Every node has a virtual visit count V(s) and every edge V(a), both 0 between steps; after
// descent j picks its path, V += 1 on every edge and node of the path and on the leaf, so later descents of the
// step see it:
//   effective counts     n_eff = N(a) + V(a), N_eff(s) = N(s) + V(s)
//   effective value sum  w_eff = V(a) > 0 ? W(a) - vl * V(a) : W(a), IEEE double, no contraction
//   uct                  the unvisited-edge draw counts edges with n_eff == 0, else uct score(w_eff, n_eff, L[N_eff(s)])
//   puct                 puct score(w_eff, n_eff, P, sqrt(N_eff(s))); a terminal child still scores its outcome
// The leaf rule is unchanged (a terminal node or N(s) == 0, real visits only), so every descent of step 0 stops
// at the root, and a descent may end at a leaf an earlier descent of the step already took (a repeated leaf, an
// ordinary row).  Backup takes rows j = 0 .. K-1 in order: row j removes its V and adds its value as before; a
// PUCT leaf is expanded by the lowest row whose leaf it is.  W only ever receives real values.
// Storage for K > 1: K paths, K (leaf slot, depth, status) entries and K*R rollout slots per tree, and a u16 V per
// node and per edge:
//   K-leaf bytes per tree = (bytes per tree of the kind above) + (K - 1) * (16 + 8*P + R * (rw*4 + 16))
//                           + S * 2 * (1 + M)
// K = 1 is exactly the search above and allocates nothing more.
#pragma once
#include <stdint.h>

#include "twixt_engine.cuh"
#include "twixt_philox.cuh"

#if !defined(__CUDA_ARCH__)
#include <cmath>
#endif

namespace twixt {

enum : int { kLeafNeedsValue = 0, kLeafTerminal = 1, kLeafSolved = 2 };

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

// the PUCT formula of the header comment above
TW_HD int64_t mcts_puct_bytes_per_tree(const MctsSizes& s) { return mcts_bytes_per_tree(s) + s.slots * 9 * s.edges; }

// the solver formulas of the header comment above
TW_HD int64_t mcts_solve_bytes_per_tree(const MctsSizes& s, bool puct) {
  return (puct ? mcts_puct_bytes_per_tree(s) : mcts_bytes_per_tree(s) + s.slots * s.edges) + 1;
}

// the K-leaf formula of the header comment above, from the bytes per tree of the search kind at K = 1
TW_HD int64_t mcts_parallel_bytes_per_tree(const MctsSizes& s, int64_t kind_bytes, int leaves_per_step) {
  if (leaves_per_step <= 1) return kind_bytes;
  return kind_bytes + static_cast<int64_t>(leaves_per_step - 1) * (16 + 8 * s.path + s.rollouts * (s.rw * 4 + 16)) +
         s.slots * 2 * (1 + s.edges);
}

// w_eff of an edge with value sum w and V(a) = v virtual visits under virtual loss vl.  Bit-identical on the
// device and on a host compiled with -ffp-contract=off; w itself when v == 0.
TW_HD double mcts_virtual_w(double w, uint32_t v, double vl) {
  if (v == 0u) return w;
#if defined(__CUDA_ARCH__)
  return __dsub_rn(w, __dmul_rn(vl, static_cast<double>(v)));
#else
  return w - vl * static_cast<double>(v);
#endif
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

// sqrt(N(s)) of the PUCT score, once per node
TW_HD double mcts_sqrt_visits(uint32_t parent_visits) {
#if defined(__CUDA_ARCH__)
  return __dsqrt_rn(static_cast<double>(parent_visits));
#else
  return std::sqrt(static_cast<double>(parent_visits));
#endif
}

// PUCT score of an edge with N(a) = n visits, value sum w and prior p under a parent with sqrt(N(s)) =
// sqrt_parent, in open_spiel's evaluation order (SearchNode.puct_value).  Bit-identical on the device and on a
// host compiled with -ffp-contract=off.
TW_HD double mcts_puct_score(double w, uint32_t n, float p, double sqrt_parent, double c) {
  const double nd = static_cast<double>(n), n1 = static_cast<double>(n) + 1.0;
#if defined(__CUDA_ARCH__)
  const double q = n > 0u ? __ddiv_rn(w, nd) : 0.0;
  const double u = __ddiv_rn(__dmul_rn(__dmul_rn(c, static_cast<double>(p)), sqrt_parent), n1);
  return __dadd_rn(q, u);
#else
  const double q = n > 0u ? w / nd : 0.0;
  const double u = ((c * static_cast<double>(p)) * sqrt_parent) / n1;
  return q + u;
#endif
}

// P(a) when no priors are given: float32(1.0 / L), RandomRolloutEvaluator.prior
TW_HD float mcts_uniform_prior(int legal) {
#if defined(__CUDA_ARCH__)
  return __double2float_rn(__ddiv_rn(1.0, static_cast<double>(legal)));
#else
  return static_cast<float>(1.0 / static_cast<double>(legal));
#endif
}

// the tie key of edge `edge` of node slot `slot` (its place in open_spiel's shuffled child list)
TW_HD uint32_t mcts_tie_key(uint64_t seed, uint32_t tree_stream, uint32_t slot, uint32_t edge) {
  uint32_t r[4];
  philox4x32_10(tree_stream, slot, edge, 2u, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), r);
  return r[0];
}

// PUCT selection: (score a, key ka, edge ia) beats (b, kb, ib): the larger score, then the smaller key, then
// the lower edge
TW_HD bool mcts_puct_beats(double a, uint32_t ka, int ia, double b, uint32_t kb, int ib) {
  if (a != b) return a > b;
  if (ka != kb) return ka < kb;
  return ia < ib;
}

// terminal outcome byte of an edge: 0 while its child does not exist or is not terminal, else
// 2 + Returns()[player to move at the parent]
TW_HD uint8_t mcts_outcome_code(const Header& child, int player) {
  const int red = child.result == kRedWin ? 1 : (child.result == kBlueWin ? -1 : 0);
  return static_cast<uint8_t>(2 + (player == 0 ? red : -red));
}
TW_HD int mcts_outcome_value(uint8_t code) { return code == 0 ? 0 : static_cast<int>(code) - 2; }

// MCTS-Solver proof step of an expanded node from its L > 0 edge codes, given their maximum and whether every one
// is non-zero: the node is proven when some edge is a win for its player to move (code 3) or every edge is
// proven.  Returns its value v for that player, or kUnproven.
enum : int { kUnproven = -128 };
TW_HD int mcts_proven_value(int max_code, bool all_proven) {
  return (max_code == 3 || all_proven) ? max_code - 2 : static_cast<int>(kUnproven);
}
// the code of the parent's edge into a node proven with value v (zero-sum, players alternate by ply)
TW_HD uint8_t mcts_parent_code(int v) { return static_cast<uint8_t>(2 - v); }

// PUCT BestChild (open_spiel SearchNode.sort_key): (outcome value, N, W), then the smaller key, then the
// lower edge
TW_HD bool mcts_puct_best_beats(int oa, uint32_t na, double wa, uint32_t ka, int ia, int ob, uint32_t nb, double wb,
                                uint32_t kb, int ib) {
  if (oa != ob) return oa > ob;
  if (na != nb) return na > nb;
  if (wa != wb) return wa > wb;
  if (ka != kb) return ka < kb;
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
