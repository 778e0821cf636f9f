// TEST-ONLY: the Gumbel AlphaZero search of twixt_mcts.cu restated for the HOST on the product's helpers
// (twixt_for_open_spiel_b200/csrc/twixt_mcts.cuh: mcts_exp, the completed-Q pieces, the scores, mcts_lane_sums,
// mcts_considered_visits), the rules (twixt_engine.cuh) and the Philox stream, built with -ffp-contract=off, so that
// `pytest -m "not gpu"` can compare it node for node with the executable specification (tests/gumbel_spec.py)
// without a GPU.  The storage mirrors the device arena (creation-order slots, ascending edges, N / W / child /
// logit per edge, v per node).  It is stepwise -- select, then backup with optional values and logits.  This file
// is never part of libtwixt_b200.so.
#include <cstdint>
#include <cstring>
#include <vector>

#include "twixt_engine.cuh"
#include "twixt_mcts.cuh"
#include "twixt_philox.cuh"

using namespace twixt;
using Rec = RecordRef<1>;

namespace {

constexpr int kStack = 48;

// twixt_playout's policy on one record (as tests/mcts_harness.cc), played to the end
void host_playout(uint32_t* rec, int n, uint64_t seed, uint64_t stream) {
  Rec b{rec, n};
  Header h;
  load_header(b, h);
  int step = 0;
  uint32_t r[4] = {0, 0, 0, 0};
  while (h.result == kOpen) {
    if ((step & 3) == 0)
      philox4x32_10(static_cast<uint32_t>(stream), static_cast<uint32_t>(stream >> 32), static_cast<uint32_t>(step) >> 2,
                    0u, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), r);
    const int k = static_cast<int>(playout_index(r[step & 3], static_cast<uint32_t>(legal_count(h, n))));
    int x, y;
    select_legal(b, h, k, x, y);
    apply_legal_cell<kStack>(b, h, x, y);
    ++step;
  }
  store_header(b, h);
}

Header header_of(const uint32_t* rec) {
  Header h;
  unpack_header(rec[0], rec[1], rec[2], rec[3], h);
  return h;
}

struct Tree {
  int n, rw, M, S, R, nodes = 1, k = 0, mc, cols;
  uint64_t seed;
  uint32_t T;
  double c_visit, c_scale;
  std::vector<uint32_t> recs;
  std::vector<int32_t> parent, action, legal, child, table;
  std::vector<uint32_t> node_n, edge_n;
  std::vector<uint16_t> edge_action;
  std::vector<double> edge_w, node_value;
  std::vector<float> edge_logit, gumbel;
  std::vector<int> path_node, path_edge;
  int leaf = -1;
};

// what gumbel_node computes on the device
struct NodeQ {
  double max_logit, v_mix, q_min, q_max, scale;
  uint32_t sum_n, max_n;
};

NodeQ node_q(const Tree& t, int node) {
  const size_t e0 = static_cast<size_t>(node) * t.M;
  const int L = t.legal[node];
  NodeQ s;
  s.max_logit = -INFINITY;
  s.sum_n = 0u;
  s.max_n = 0u;
  for (int i = 0; i < L; ++i) {
    s.max_logit = mcts_max(s.max_logit, static_cast<double>(t.edge_logit[e0 + i]));
    s.sum_n += t.edge_n[e0 + i];
    s.max_n = t.edge_n[e0 + i] > s.max_n ? t.edge_n[e0 + i] : s.max_n;
  }
  double weighted_q = 0.0;
  if (s.sum_n > 0u) {
    auto e = [&](int i) { return mcts_exp(static_cast<double>(t.edge_logit[e0 + i]) - s.max_logit); };
    auto visited = [&](int i) { return t.edge_n[e0 + i] > 0u; };
    const double z = mcts_lane_sums(L, e, [](int) { return true; });
    const double sp = mcts_lane_sums(L, [&](int i) { return mcts_gumbel_prob(e(i), z); }, visited);
    weighted_q = mcts_lane_sums(
        L, [&](int i) { return mcts_gumbel_mix_term(mcts_gumbel_prob(e(i), z), t.edge_w[e0 + i], t.edge_n[e0 + i], sp); },
        visited);
  }
  s.v_mix = mcts_gumbel_mixed_value(t.node_value[node], s.sum_n, weighted_q);
  s.q_min = INFINITY;
  s.q_max = -INFINITY;
  for (int i = 0; i < L; ++i) {
    const double q = mcts_gumbel_completed_q(t.edge_w[e0 + i], t.edge_n[e0 + i], s.v_mix);
    s.q_min = mcts_min(s.q_min, q);
    s.q_max = mcts_max(s.q_max, q);
  }
  s.scale = mcts_gumbel_scale(t.c_visit, t.c_scale, s.max_n);
  return s;
}

double sigma_of(const Tree& t, const NodeQ& s, size_t e) {
  return mcts_gumbel_sigma(mcts_gumbel_completed_q(t.edge_w[e], t.edge_n[e], s.v_mix), s.q_min, s.q_max, s.scale);
}

// softmax(l + sigma) = e(i) / z: returns z and the max of l + sigma
void softmax_norm(const Tree& t, int node, const NodeQ& s, double& mx, double& z) {
  const size_t e0 = static_cast<size_t>(node) * t.M;
  const int L = t.legal[node];
  mx = -INFINITY;
  for (int i = 0; i < L; ++i) mx = mcts_max(mx, static_cast<double>(t.edge_logit[e0 + i]) + sigma_of(t, s, e0 + i));
  const double m = mx;
  z = mcts_lane_sums(
      L, [&](int i) { return mcts_exp((static_cast<double>(t.edge_logit[e0 + i]) + sigma_of(t, s, e0 + i)) - m); },
      [](int) { return true; });
}

int root_argmax(const Tree& t, const NodeQ& s, int64_t considered) {
  int bi = -1;
  double best = 0.0;
  for (int i = 0; i < t.legal[0]; ++i) {
    if (static_cast<int64_t>(t.edge_n[i]) != considered) continue;
    const double sc = mcts_gumbel_root_score(t.gumbel[t.edge_action[i]], t.edge_logit[i], s.max_logit, sigma_of(t, s, i));
    if (bi < 0 || mcts_score_beats(sc, i, best, bi)) {
      best = sc;
      bi = i;
    }
  }
  return bi < 0 ? 0 : bi;
}

}  // namespace

extern "C" {

double gh_exp(double x) { return mcts_exp(x); }

void gh_considered_visits(int m, int num_simulations, int32_t* out) { mcts_considered_visits(m, num_simulations, out); }

int64_t gh_bytes_per_tree(int n, int max_simulations, int n_rollouts) {
  return mcts_gumbel_bytes_per_tree(mcts_sizes(n, max_simulations, n_rollouts), static_cast<int64_t>(n) * n);
}

// gumbel: [n*n] float32 root noise (nullable: 0)
void* gh_create(const uint32_t* root_rec, int n, uint64_t seed, uint32_t tree_stream, int R, int sims,
                int max_considered, double c_visit, double c_scale, const float* gumbel) {
  const MctsSizes s = mcts_sizes(n, sims, R);
  Tree* t = new Tree();
  t->n = n;
  t->rw = static_cast<int>(s.rw);
  t->M = static_cast<int>(s.edges);
  t->S = static_cast<int>(s.slots);
  t->R = R;
  t->seed = seed;
  t->T = tree_stream;
  t->c_visit = c_visit;
  t->c_scale = c_scale;
  t->mc = max_considered < t->M ? max_considered : t->M;
  t->cols = sims - 1;
  t->table.assign(static_cast<size_t>(t->mc + 1) * t->cols, 0);
  for (int m = 0; m <= t->mc; ++m) mcts_considered_visits(m, t->cols, t->table.data() + static_cast<size_t>(m) * t->cols);
  const size_t S = t->S, E = S * t->M;
  t->recs.assign(S * t->rw, 0u);
  t->parent.assign(S, -1);
  t->action.assign(S, -1);
  t->legal.assign(S, -1);
  t->node_n.assign(S, 0u);
  t->node_value.assign(S, 0.0);
  t->child.assign(E, -1);
  t->edge_n.assign(E, 0u);
  t->edge_action.assign(E, 0);
  t->edge_w.assign(E, 0.0);
  t->edge_logit.assign(E, 0.0f);
  t->gumbel.assign(static_cast<size_t>(n) * n, 0.0f);
  if (gumbel != nullptr) std::memcpy(t->gumbel.data(), gumbel, t->gumbel.size() * sizeof(float));
  std::memcpy(t->recs.data(), root_rec, t->rw * sizeof(uint32_t));
  return t;
}

void gh_destroy(void* h) { delete static_cast<Tree*>(h); }

// descends as mcts_gumbel_select_kernel; writes the leaf record to leaf_out (nullable), returns 1 for a terminal
// leaf, else 0
int gh_select(void* h, uint32_t* leaf_out) {
  Tree& t = *static_cast<Tree*>(h);
  t.path_node.clear();
  t.path_edge.clear();
  int node = 0;
  for (;;) {
    uint32_t* rec = &t.recs[static_cast<size_t>(node) * t.rw];
    const Header hd = header_of(rec);
    if (hd.result != kOpen || t.node_n[node] == 0) break;
    const size_t e0 = static_cast<size_t>(node) * t.M;
    const NodeQ s = node_q(t, node);
    int edge;
    if (node == 0) {
      const int m = t.mc < t.legal[0] ? t.mc : t.legal[0];
      const int64_t considered =
          static_cast<int>(s.sum_n) < t.cols ? t.table[static_cast<size_t>(m) * t.cols + s.sum_n] : -1;
      edge = root_argmax(t, s, considered);
    } else {
      double mx, z;
      softmax_norm(t, node, s, mx, z);
      edge = -1;
      double best = 0.0;
      for (int i = 0; i < t.legal[node]; ++i) {
        const double e = mcts_exp((static_cast<double>(t.edge_logit[e0 + i]) + sigma_of(t, s, e0 + i)) - mx);
        const double sc = mcts_gumbel_interior_score(e, z, t.edge_n[e0 + i], s.sum_n);
        if (edge < 0 || mcts_score_beats(sc, i, best, edge)) {
          best = sc;
          edge = i;
        }
      }
    }
    t.path_node.push_back(node);
    t.path_edge.push_back(edge);
    if (t.child[e0 + edge] < 0) {
      const int ch = t.nodes++;
      uint32_t* crec = &t.recs[static_cast<size_t>(ch) * t.rw];
      std::memcpy(crec, rec, t.rw * sizeof(uint32_t));
      Rec cb{crec, t.n};
      Header chh = hd;
      const int a = t.edge_action[e0 + edge];
      apply_legal_cell<kStack>(cb, chh, a / t.n, a % t.n);
      store_header(cb, chh);
      t.parent[ch] = node;
      t.action[ch] = a;
      t.child[e0 + edge] = ch;
    }
    node = t.child[e0 + edge];
  }
  t.leaf = node;
  const uint32_t* lr = &t.recs[static_cast<size_t>(node) * t.rw];
  if (leaf_out != nullptr) std::memcpy(leaf_out, lr, t.rw * sizeof(uint32_t));
  return header_of(lr).result != kOpen ? 1 : 0;
}

// backs up as mcts_gumbel_backup_kernel: values [2] (nullptr: the mean of R host rollouts), logits [n*n] (nullptr:
// 0); v(leaf) is the value for its player to move and a non-terminal leaf is expanded with the logits
void gh_backup(void* h, const float* values, const float* logits) {
  Tree& t = *static_cast<Tree*>(h);
  const int node = t.leaf;
  uint32_t* leaf = &t.recs[static_cast<size_t>(node) * t.rw];
  const Header lh = header_of(leaf);
  double v[2];
  if (lh.result != kOpen) {
    mcts_terminal_value(lh, v);
  } else if (values != nullptr) {
    v[0] = static_cast<double>(values[0]);
    v[1] = static_cast<double>(values[1]);
  } else {
    std::vector<uint32_t> roll(t.rw);
    double s0 = 0.0, s1 = 0.0;
    for (int r = 0; r < t.R; ++r) {
      std::memcpy(roll.data(), leaf, t.rw * sizeof(uint32_t));
      host_playout(roll.data(), t.n, t.seed,
                   mcts_rollout_stream(t.T, static_cast<uint32_t>(t.k), static_cast<uint32_t>(t.R), static_cast<uint32_t>(r)));
      double ret[2];
      mcts_terminal_value(header_of(roll.data()), ret);
      s0 += ret[0];
      s1 += ret[1];
    }
    v[0] = s0 / t.R;
    v[1] = s1 / t.R;
  }
  for (size_t i = 0; i < t.path_node.size(); ++i) {
    const int p = t.path_node[i];
    const size_t e = static_cast<size_t>(p) * t.M + t.path_edge[i];
    t.node_n[p] += 1;
    t.edge_n[e] += 1;
    t.edge_w[e] += v[header_of(&t.recs[static_cast<size_t>(p) * t.rw]).ply & 1u];
  }
  t.node_n[node] += 1;
  t.node_value[node] = v[lh.ply & 1u];
  if (lh.result == kOpen) {
    const size_t e0 = static_cast<size_t>(node) * t.M;
    Rec b{leaf, t.n};
    int L = 0;
    for (int x = 0; x < t.n; ++x) {
      uint32_t w = legal_word(b, lh, x);
      while (w) {
        const int y = tw_ctz(w);
        w &= w - 1u;
        t.edge_action[e0 + L] = static_cast<uint16_t>(x * t.n + y);
        ++L;
      }
    }
    for (int i = 0; i < L; ++i) {
      t.edge_n[e0 + i] = 0;
      t.edge_w[e0 + i] = 0.0;
      t.child[e0 + i] = -1;
      t.edge_logit[e0 + i] = logits != nullptr ? logits[t.edge_action[e0 + i]] : 0.0f;
    }
    t.legal[node] = L;
  }
  t.k += 1;
}

// Per node slot (creation order): parent slot, action from the parent, N(s), edge count (-1 unexpanded), v(s) and
// [slots, M] edge visits / value sums / logits in ascending action order.  Returns the number of nodes.
int gh_dump(void* h, int32_t* node_parent, int32_t* node_action, uint32_t* node_n, int32_t* node_legal,
            double* node_value, uint32_t* edge_n, double* edge_w, float* edge_logit) {
  Tree& t = *static_cast<Tree*>(h);
  for (int s = 0; s < t.nodes; ++s) {
    node_parent[s] = t.parent[s];
    node_action[s] = t.action[s];
    node_n[s] = t.node_n[s];
    node_legal[s] = t.legal[s];
    node_value[s] = t.node_value[s];
    for (int i = 0; i < (t.legal[s] > 0 ? t.legal[s] : 0); ++i) {
      const size_t e = static_cast<size_t>(s) * t.M + i;
      edge_n[e] = t.edge_n[e];
      edge_w[e] = t.edge_w[e];
      edge_logit[e] = t.edge_logit[e];
    }
  }
  return t.nodes;
}

// as mcts_gumbel_stats_kernel: the action (-1: unexpanded root) and the improved policy [n*n]
void gh_stats(void* h, int32_t* out_action, float* out_policy) {
  Tree& t = *static_cast<Tree*>(h);
  std::memset(out_policy, 0, static_cast<size_t>(t.n) * t.n * sizeof(float));
  if (t.legal[0] < 0) {
    *out_action = -1;
    return;
  }
  const NodeQ s = node_q(t, 0);
  *out_action = t.edge_action[root_argmax(t, s, s.max_n)];
  double mx, z;
  softmax_norm(t, 0, s, mx, z);
  for (int i = 0; i < t.legal[0]; ++i)
    out_policy[t.edge_action[i]] =
        static_cast<float>(mcts_exp((static_cast<double>(t.edge_logit[i]) + sigma_of(t, s, i)) - mx) / z);
}

}  // extern "C"
