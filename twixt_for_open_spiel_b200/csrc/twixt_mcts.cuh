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
//
// Tree reuse (twixt_mcts_advance(actions, keep_nodes)): the child of the root along actions[t] becomes the new
// root.  The kept nodes are that child's subtree, renumbered by their rank in old slot order (the new root is slot
// 0, children stay above their parents), and only the first keep_nodes of that order are kept; an edge whose child
// the cap drops goes back to N = 0, W = 0, child -1 (prior, tie key and outcome code stay).  Every kept node keeps
// its record, N(s), legal count and its edges' action, N, W, prior, tie key and outcome code, children remapped.
// A legal action without a child clears the tree to the root with the move applied; -1 keeps the root and only
// applies the cap; an illegal action leaves the tree as it is.  A solver search's new root takes code 4 - c from
// the chosen edge's code c != 0 (the child's value for its own player to move), else 0.  The draw and rollout
// streams keep counting k: a tree never repeats a Philox counter.  The kernel needs an int32 old -> new slot map of
// S entries per tree, allocated at the first advance.
//
// Gumbel AlphaZero (twixt_mcts_create_gumbel; mctx gumbel_muzero_policy, Danihelka et al., ICLR 2022): the tree
// above, one node per simulation, leaves expanded at their backup as PUCT does, but every edge carries a float32
// logit l(a) (the caller's [n*n] row, 0 without one) and every node its raw value v(s) (its evaluation for its own
// player to move), and the root takes Gumbel noise g(a) per action cell.  Selection (IEEE double, no
// contraction, the helpers below):
//   pi(a)      max(softmax(l)(a), smallest normal double)
//   v_mix      (v + SN * sum_{N(b)>0} (pi(b) * q(b) / sum_{N(b)>0} pi(b))) / (SN + 1),  q = W/N, SN = sum N(b)
//   q~(a)      q(a) if N(a) > 0, else v_mix;  q^ = (q~ - min q~) / max(max q~ - min q~, 1e-8)
//   sigma(a)   ((c_visit + max N(b)) * c_scale) * q^(a)
//   interior   argmax of softmax(l + sigma)(a) - N(a) / (1 + SN), ties to the lower edge
//   root       Sequential Halving: among edges with N(a) = table[min(max_considered, L)][SN], argmax of
//              max(-1e9, (g(a) + (l(a) - max l)) + sigma(a)), ties to the lower edge (none eligible: edge 0)
//   action     the root score among the edges with N(a) = max N;  improved policy softmax(l + sigma) at the root
// table is mctx's get_table_of_considered_visits(max_considered, max_simulations - 1) (mcts_considered_visits).
// Every exp is mcts_exp and every sum over a node's edges is in the order of mcts_lane_sums: lane l adds edges
// l, l+32, .. from 0.0, then an xor butterfly over offsets 16, 8, 4, 2, 1.  A Gumbel search has no priors, tie keys
// or outcome bytes; it adds 4 (logit f32) per edge, 8 (v f64) per node and 4*n*n (root noise f32) per tree:
//   Gumbel bytes per tree = S * (rw*4 + 16 + 22*M) + 16 + 8*P + R * (rw*4 + 16) + 4*n*n
// plus the table, (min(max_considered, M) + 1) * (max_simulations - 1) int32, once per search.
#pragma once
#include <stdint.h>

#include "twixt_engine.cuh"
#include "twixt_philox.cuh"

#include <cstring>
#include <vector>
#if !defined(__CUDA_ARCH__)
#include <cmath>
#endif

namespace twixt {

enum : int { kLeafNeedsValue = 0, kLeafTerminal = 1, kLeafSolved = 2 };
// statuses of twixt_mcts_advance: the new root kept its statistics (N(root) > 0), the action was illegal (tree
// unchanged), the new root has none (N(root) == 0: the next simulation evaluates it)
enum : int { kRootKept = 0, kRootIllegal = 1, kRootFresh = 2 };

// the solver root code of a tree advanced along an edge with outcome code c (twixt_mcts_advance)
TW_HD uint8_t mcts_advanced_root_code(uint8_t c) { return c != 0 ? static_cast<uint8_t>(4 - c) : 0; }

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

// ------------------------------------------------------------------------------------ Gumbel AlphaZero ---
// IEEE double operations, round to nearest, identical on the device and on a host built with -ffp-contract=off
TW_HD double mcts_add(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
TW_HD double mcts_sub(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dsub_rn(a, b);
#else
  return a - b;
#endif
}
TW_HD double mcts_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
TW_HD double mcts_div(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}
TW_HD double mcts_max(double a, double b) { return a > b ? a : b; }
TW_HD double mcts_min(double a, double b) { return a < b ? a : b; }

// 2^j for -1022 <= j <= 1023, exact
TW_HD double mcts_pow2(int j) {
  const uint64_t bits = static_cast<uint64_t>(j + 1023) << 52;
#if defined(__CUDA_ARCH__)
  return __longlong_as_double(static_cast<long long>(bits));
#else
  double d;
  std::memcpy(&d, &bits, sizeof(d));
  return d;
#endif
}

// exp(x) for x <= 0 (every softmax argument is max-centred), part of the specification: 0 below -746 (and for NaN);
// else k = round-half-even(x * log2(e)), r = (x - k*ln2_hi) - k*ln2_lo (Cody-Waite; k*ln2_hi is exact), the
// degree-13 Taylor polynomial of e^r in Horner form (coefficients float64(1/j!)), scaled by 2^(k >> 1) and then
// 2^(k - (k >> 1)): only the last product can round (a subnormal result).  Within 1 ulp of a correctly rounded exp.
TW_HD double mcts_exp_step(double p, double r, double c) { return mcts_add(mcts_mul(p, r), c); }
TW_HD double mcts_exp(double x) {
  if (!(x >= -746.0)) return 0.0;
#if defined(__CUDA_ARCH__)
  const int k = __double2int_rn(__dmul_rn(x, 0x1.71547652b82fep+0));
#else
  const int k = static_cast<int>(std::nearbyint(x * 0x1.71547652b82fep+0));
#endif
  const double kd = static_cast<double>(k);
  const double r = mcts_sub(mcts_sub(x, mcts_mul(kd, 0x1.62e42fee00000p-1)), mcts_mul(kd, 0x1.a39ef35793c76p-33));
  double p = 0x1.6124613a86d09p-33;             // 1/13!
  p = mcts_exp_step(p, r, 0x1.1eed8eff8d898p-29);  // 1/12!
  p = mcts_exp_step(p, r, 0x1.ae64567f544e4p-26);  // 1/11!
  p = mcts_exp_step(p, r, 0x1.27e4fb7789f5cp-22);  // 1/10!
  p = mcts_exp_step(p, r, 0x1.71de3a556c734p-19);  // 1/9!
  p = mcts_exp_step(p, r, 0x1.a01a01a01a01ap-16);  // 1/8!
  p = mcts_exp_step(p, r, 0x1.a01a01a01a01ap-13);  // 1/7!
  p = mcts_exp_step(p, r, 0x1.6c16c16c16c17p-10);  // 1/6!
  p = mcts_exp_step(p, r, 0x1.1111111111111p-7);   // 1/5!
  p = mcts_exp_step(p, r, 0x1.5555555555555p-5);   // 1/4!
  p = mcts_exp_step(p, r, 0x1.5555555555555p-3);   // 1/3!
  p = mcts_exp_step(p, r, 0x1.0p-1);
  p = mcts_exp_step(p, r, 1.0);
  p = mcts_exp_step(p, r, 1.0);
  return mcts_mul(mcts_mul(p, mcts_pow2(k >> 1)), mcts_pow2(k - (k >> 1)));
}

// pi(a) from e = mcts_exp(l(a) - max l) and Z = the sum of e: raised to the smallest normal double (mctx's
// jnp.finfo.tiny in _compute_mixed_value)
TW_HD double mcts_gumbel_prob(double e, double z) { return mcts_max(mcts_div(e, z), 0x1.0p-1022); }
// one term of the mixed value's weighted Q: pi(b) * q(b) / sum_{N(b)>0} pi(b), q = W/N
TW_HD double mcts_gumbel_mix_term(double pi, double w, uint32_t n, double sum_probs) {
  return mcts_div(mcts_mul(pi, mcts_div(w, static_cast<double>(n))), sum_probs);
}
// v_mix from the node's raw value, SN = sum N(b) and the weighted Q
TW_HD double mcts_gumbel_mixed_value(double raw, uint32_t sum_n, double weighted_q) {
  const double sn = static_cast<double>(sum_n);
  return mcts_div(mcts_add(raw, mcts_mul(sn, weighted_q)), mcts_add(sn, 1.0));
}
// q~(a): W/N for a visited edge, else v_mix
TW_HD double mcts_gumbel_completed_q(double w, uint32_t n, double v_mix) {
  return n > 0u ? mcts_div(w, static_cast<double>(n)) : v_mix;
}
// (c_visit + max N(b)) * c_scale, the factor of sigma
TW_HD double mcts_gumbel_scale(double c_visit, double c_scale, uint32_t max_n) {
  return mcts_mul(mcts_add(c_visit, static_cast<double>(max_n)), c_scale);
}
// sigma(a) from q~(a), the node's min and max q~ and its scale
TW_HD double mcts_gumbel_sigma(double q, double q_min, double q_max, double scale) {
  return mcts_mul(scale, mcts_div(mcts_sub(q, q_min), mcts_max(mcts_sub(q_max, q_min), 1e-8)));
}
// interior score pi'(a) - N(a) / (1 + SN), pi'(a) = e / Z' (e = mcts_exp(l + sigma - max(l + sigma)))
TW_HD double mcts_gumbel_interior_score(double e, double z, uint32_t n, uint32_t sum_n) {
  return mcts_sub(mcts_div(e, z), mcts_div(static_cast<double>(n), mcts_add(static_cast<double>(sum_n), 1.0)));
}
// root score max(-1e9, (g + (l - max l)) + sigma)
TW_HD double mcts_gumbel_root_score(float g, float logit, double max_logit, double sigma) {
  return mcts_max(-1e9, mcts_add(mcts_add(static_cast<double>(g), mcts_sub(static_cast<double>(logit), max_logit)),
                                 sigma));
}

// The device's order of a sum over L edges, on the host (host code only): lane l adds terms l, l+32, .. (ascending) from 0.0 where
// include(i), then partials combine as p[l] + p[l ^ d] for d = 16, 8, 4, 2, 1 (the same in every lane).
template <class Term, class Include>
double mcts_lane_sums(int L, Term term, Include include) {
  double p[32];
  for (int l = 0; l < 32; ++l) {
    p[l] = 0.0;
    for (int i = l; i < L; i += 32)
      if (include(i)) p[l] = p[l] + term(i);
  }
  for (int d = 16; d > 0; d >>= 1) {
    double q[32];
    for (int l = 0; l < 32; ++l) q[l] = p[l] + p[l ^ d];
    std::memcpy(p, q, sizeof(p));
  }
  return p[0];
}

// mctx seq_halving.get_sequence_of_considered_visits(m, num_simulations) in integer arithmetic: out[0 ..
// num_simulations) (host code only)
inline void mcts_considered_visits(int m, int num_simulations, int32_t* out) {
  if (m <= 1) {
    for (int i = 0; i < num_simulations; ++i) out[i] = i;
    return;
  }
  int log2max = 0;  // ceil(log2(m))
  while ((1 << log2max) < m) ++log2max;
  std::vector<int32_t> visits(static_cast<size_t>(m), 0);
  int num_considered = m, len = 0;
  while (len < num_simulations) {
    int extra = num_simulations / (log2max * num_considered);
    if (extra < 1) extra = 1;
    for (int e = 0; e < extra; ++e) {
      for (int i = 0; i < num_considered; ++i, ++len)
        if (len < num_simulations) out[len] = visits[i];
      for (int i = 0; i < num_considered; ++i) visits[i] += 1;
    }
    num_considered = num_considered / 2 > 2 ? num_considered / 2 : 2;
  }
}

// the Gumbel formula of the header comment above; cells = n*n
TW_HD int64_t mcts_gumbel_bytes_per_tree(const MctsSizes& s, int64_t cells) {
  return mcts_bytes_per_tree(s) + s.slots * (8 + 4 * s.edges) + 4 * cells;
}

}  // namespace twixt
