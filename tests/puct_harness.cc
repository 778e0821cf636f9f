// TEST-ONLY: the PUCT search of twixt_mcts.cu restated for the HOST on the product's helpers
// (twixt_for_open_spiel_b200/csrc/twixt_mcts.cuh: score, tie key, outcome byte, BestChild, uniform prior), the
// rules (twixt_engine.cuh) and the Philox stream, built with -ffp-contract=off, so that `pytest -m "not gpu"`
// can compare it node for node with the executable specification (tests/puct_spec.py) without a GPU.  The
// storage mirrors the device arena (creation-order slots, ascending edges, N / W / child / P / key / outcome
// per edge).  It is stepwise -- select, then backup with optional values and priors -- so that the tests can
// drive it with host rollouts or with stand-in priors and values.  This file is never part of libtwixt_b200.so.
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
  int n, rw, M, S, R, nodes = 1, k = 0;
  uint64_t seed;
  uint32_t T;
  double c;
  std::vector<uint32_t> recs;
  std::vector<int32_t> parent, action, legal, child;
  std::vector<uint32_t> node_n, edge_n, edge_key;
  std::vector<uint16_t> edge_action;
  std::vector<double> edge_w;
  std::vector<float> edge_p;
  std::vector<uint8_t> edge_out;
  std::vector<int> path_node, path_edge;
  int leaf = -1;
};

}  // namespace

extern "C" {

double ph_score(double w, uint32_t n, float p, uint32_t parent_visits, double c) {
  return mcts_puct_score(w, n, p, mcts_sqrt_visits(parent_visits), c);
}

uint32_t ph_tie_key(uint64_t seed, uint32_t tree_stream, uint32_t slot, uint32_t edge) {
  return mcts_tie_key(seed, tree_stream, slot, edge);
}

int64_t ph_bytes_per_tree(int n, int max_simulations, int n_rollouts) {
  return mcts_puct_bytes_per_tree(mcts_sizes(n, max_simulations, n_rollouts));
}

void* ph_create(const uint32_t* root_rec, int n, uint64_t seed, uint32_t tree_stream, int R, double c, int sims) {
  const MctsSizes s = mcts_sizes(n, sims, R);
  Tree* t = new Tree();
  t->n = n;
  t->rw = static_cast<int>(s.rw);
  t->M = static_cast<int>(s.edges);
  t->S = static_cast<int>(s.slots);
  t->R = R;
  t->seed = seed;
  t->T = tree_stream;
  t->c = c;
  const size_t S = t->S, E = S * t->M;
  t->recs.assign(S * t->rw, 0u);
  t->parent.assign(S, -1);
  t->action.assign(S, -1);
  t->legal.assign(S, -1);
  t->node_n.assign(S, 0u);
  t->child.assign(E, -1);
  t->edge_n.assign(E, 0u);
  t->edge_key.assign(E, 0u);
  t->edge_action.assign(E, 0);
  t->edge_w.assign(E, 0.0);
  t->edge_p.assign(E, 0.0f);
  t->edge_out.assign(E, 0);
  std::memcpy(t->recs.data(), root_rec, t->rw * sizeof(uint32_t));
  return t;
}

void ph_destroy(void* h) { delete static_cast<Tree*>(h); }

// descends as mcts_select_kernel<true>; writes the leaf record to leaf_out (nullable), returns 1 for a terminal
// leaf, else 0
int ph_select(void* h, uint32_t* leaf_out) {
  Tree& t = *static_cast<Tree*>(h);
  t.path_node.clear();
  t.path_edge.clear();
  int node = 0;
  for (;;) {
    uint32_t* rec = &t.recs[static_cast<size_t>(node) * t.rw];
    const Header hd = header_of(rec);
    if (hd.result != kOpen || t.node_n[node] == 0) break;
    const size_t e0 = static_cast<size_t>(node) * t.M;
    const double sq = mcts_sqrt_visits(t.node_n[node]);
    int edge = -1;
    double bs = 0.0;
    uint32_t bk = 0u;
    for (int i = 0; i < t.legal[node]; ++i) {
      const uint8_t o = t.edge_out[e0 + i];
      const double sc = o != 0 ? static_cast<double>(mcts_outcome_value(o))
                               : mcts_puct_score(t.edge_w[e0 + i], t.edge_n[e0 + i], t.edge_p[e0 + i], sq, t.c);
      if (edge < 0 || mcts_puct_beats(sc, t.edge_key[e0 + i], i, bs, bk, edge)) {
        bs = sc;
        bk = t.edge_key[e0 + i];
        edge = i;
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
      if (chh.result != kOpen) t.edge_out[e0 + edge] = mcts_outcome_code(chh, static_cast<int>(hd.ply & 1u));
    }
    node = t.child[e0 + edge];
  }
  t.leaf = node;
  const uint32_t* lr = &t.recs[static_cast<size_t>(node) * t.rw];
  if (leaf_out != nullptr) std::memcpy(leaf_out, lr, t.rw * sizeof(uint32_t));
  return header_of(lr).result != kOpen ? 1 : 0;
}

// backs up as mcts_backup_kernel: values [2] (nullptr: the mean of R host rollouts), priors [n*n] (nullptr:
// uniform); a non-terminal leaf is expanded with the priors
void ph_backup(void* h, const float* values, const float* priors) {
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
    const float uniform = mcts_uniform_prior(L);
    for (int i = 0; i < L; ++i) {
      t.edge_n[e0 + i] = 0;
      t.edge_w[e0 + i] = 0.0;
      t.child[e0 + i] = -1;
      t.edge_p[e0 + i] = priors != nullptr ? priors[t.edge_action[e0 + i]] : uniform;
      t.edge_key[e0 + i] = mcts_tie_key(t.seed, t.T, static_cast<uint32_t>(node), static_cast<uint32_t>(i));
      t.edge_out[e0 + i] = 0;
    }
    t.legal[node] = L;
  }
  t.k += 1;
}

// Per node slot (creation order): parent slot, action from the parent, N(s), edge count (-1 unexpanded) and
// [slots, M] edge visits / value sums / priors in ascending action order.  Returns the number of nodes; *best
// receives the root's BestChild action as mcts_root_stats_kernel (-1 while no root edge has a visit).
int ph_dump(void* h, int32_t* node_parent, int32_t* node_action, uint32_t* node_n, int32_t* node_legal,
            uint32_t* edge_n, double* edge_w, float* edge_p, int32_t* best) {
  Tree& t = *static_cast<Tree*>(h);
  for (int s = 0; s < t.nodes; ++s) {
    node_parent[s] = t.parent[s];
    node_action[s] = t.action[s];
    node_n[s] = t.node_n[s];
    node_legal[s] = t.legal[s];
    for (int i = 0; i < (t.legal[s] > 0 ? t.legal[s] : 0); ++i) {
      const size_t e = static_cast<size_t>(s) * t.M + i;
      edge_n[e] = t.edge_n[e];
      edge_w[e] = t.edge_w[e];
      edge_p[e] = t.edge_p[e];
    }
  }
  int bi = -1;
  uint32_t nmax = 0;
  for (int i = 0; i < (t.legal[0] > 0 ? t.legal[0] : 0); ++i) {
    nmax = t.edge_n[i] > nmax ? t.edge_n[i] : nmax;
    if (bi < 0 || mcts_puct_best_beats(mcts_outcome_value(t.edge_out[i]), t.edge_n[i], t.edge_w[i], t.edge_key[i], i,
                                       mcts_outcome_value(t.edge_out[bi]), t.edge_n[bi], t.edge_w[bi],
                                       t.edge_key[bi], bi))
      bi = i;
  }
  *best = nmax > 0 ? t.edge_action[bi] : -1;
  return t.nodes;
}

}  // extern "C"
