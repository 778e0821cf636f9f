// TEST-ONLY: the MCTS-Solver searches of twixt_mcts.cu (mcts_select_kernel<kPuct, true>,
// mcts_backup_kernel<true>, mcts_root_stats_kernel<true>) restated for the HOST on the product's helpers
// (twixt_for_open_spiel_b200/csrc/twixt_mcts.cuh: scores, draw, tie key, outcome codes, proof step, BestChild), the
// rules (twixt_engine.cuh) and the Philox stream, built with -ffp-contract=off, so that `pytest -m "not gpu"` can
// compare it node for node with the executable specification (tests/solver_spec.py) without a GPU.  One tree of
// either kind (UCT or PUCT, both with solve); the storage mirrors the device arena (creation-order slots, ascending
// edges, N / W / child / P / key / outcome code per edge, a root code per tree).  It is stepwise -- select, then
// backup with optional values and priors.  This file is never part of libtwixt_b200.so.
#include <cmath>
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
  bool puct;
  int n, rw, M, S, R, nodes = 1, k = 0;
  uint64_t seed;
  uint32_t T;
  double c;
  std::vector<uint32_t> recs;
  std::vector<int32_t> parent, action, legal, child;
  std::vector<uint32_t> node_n, edge_n, edge_key;
  std::vector<uint16_t> edge_action;
  std::vector<double> edge_w, logs;
  std::vector<float> edge_p;
  std::vector<uint8_t> edge_out;
  uint8_t root_out = 0;
  std::vector<int> path_node, path_edge;
  int leaf = -1, status = 0;
};

// the ascending legal list of node slot `node` into its edges, every N = 0, W = 0, no child, code 0
int expand(Tree& t, int node) {
  const uint32_t* rec = &t.recs[static_cast<size_t>(node) * t.rw];
  const Header h = header_of(rec);
  Rec b{const_cast<uint32_t*>(rec), t.n};
  const size_t e0 = static_cast<size_t>(node) * t.M;
  int L = 0;
  for (int x = 0; x < t.n; ++x) {
    uint32_t w = legal_word(b, h, x);
    while (w) {
      const int y = tw_ctz(w);
      w &= w - 1u;
      t.edge_action[e0 + L] = static_cast<uint16_t>(x * t.n + y);
      t.edge_n[e0 + L] = 0;
      t.edge_w[e0 + L] = 0.0;
      t.child[e0 + L] = -1;
      t.edge_out[e0 + L] = 0;
      ++L;
    }
  }
  t.legal[node] = L;
  return L;
}

}  // namespace

extern "C" {

int64_t sh_bytes_per_tree(int n, int max_simulations, int n_rollouts, int puct) {
  return mcts_solve_bytes_per_tree(mcts_sizes(n, max_simulations, n_rollouts), puct != 0);
}

int sh_proven_value(int max_code, int all_proven) { return mcts_proven_value(max_code, all_proven != 0); }
int sh_parent_code(int v) { return mcts_parent_code(v); }

void* sh_create(const uint32_t* root_rec, int n, uint64_t seed, uint32_t tree_stream, int R, double c, int sims,
                int puct) {
  const MctsSizes s = mcts_sizes(n, sims, R);
  Tree* t = new Tree();
  t->puct = puct != 0;
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
  t->logs.resize(S);
  for (size_t i = 0; i < S; ++i) t->logs[i] = std::log(static_cast<double>(i));
  std::memcpy(t->recs.data(), root_rec, t->rw * sizeof(uint32_t));
  return t;
}

void sh_destroy(void* h) { delete static_cast<Tree*>(h); }

// descends as mcts_select_kernel<puct, true>; writes the leaf record to leaf_out (nullable, untouched for a
// finished tree); returns the leaf status (0 needs a value, 1 terminal, 2 finished)
int sh_select(void* h, uint32_t* leaf_out) {
  Tree& t = *static_cast<Tree*>(h);
  t.path_node.clear();
  t.path_edge.clear();
  if (t.root_out != 0) return t.status = kLeafSolved;
  int node = 0;
  for (;;) {
    uint32_t* rec = &t.recs[static_cast<size_t>(node) * t.rw];
    const Header hd = header_of(rec);
    if (hd.result != kOpen || t.node_n[node] == 0) break;
    const size_t e0 = static_cast<size_t>(node) * t.M;
    int edge = -1;
    if (t.puct) {
      const double sq = mcts_sqrt_visits(t.node_n[node]);
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
    } else {
      const int L = t.legal[node] < 0 ? expand(t, node) : t.legal[node];
      int unvisited = 0;
      for (int i = 0; i < L; ++i) unvisited += t.edge_n[e0 + i] == 0 ? 1 : 0;
      if (unvisited > 0) {
        int j = static_cast<int>(mcts_draw(t.seed, t.T, static_cast<uint32_t>(t.k), static_cast<uint32_t>(unvisited)));
        for (int i = 0; i < L && edge < 0; ++i)
          if (t.edge_n[e0 + i] == 0 && j-- == 0) edge = i;
      } else {
        double bs = 0.0;
        for (int i = 0; i < L; ++i) {
          const uint8_t o = t.edge_out[e0 + i];
          const double sc = o != 0 ? static_cast<double>(mcts_outcome_value(o))
                                   : mcts_uct_score(t.edge_w[e0 + i], t.edge_n[e0 + i], t.logs[t.node_n[node]], t.c);
          if (edge < 0 || mcts_score_beats(sc, i, bs, edge)) {
            bs = sc;
            edge = i;
          }
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
      if (chh.result != kOpen) t.edge_out[e0 + edge] = mcts_outcome_code(chh, static_cast<int>(hd.ply & 1u));
    }
    node = t.child[e0 + edge];
  }
  t.leaf = node;
  const uint32_t* lr = &t.recs[static_cast<size_t>(node) * t.rw];
  if (leaf_out != nullptr) std::memcpy(leaf_out, lr, t.rw * sizeof(uint32_t));
  return t.status = header_of(lr).result != kOpen ? kLeafTerminal : kLeafNeedsValue;
}

// backs up as mcts_backup_kernel<true>: values [2] (nullptr: the mean of R host rollouts), priors [n*n] (nullptr:
// uniform, PUCT only); a finished tree ignores both, a terminal leaf runs the proof pass
void sh_backup(void* h, const float* values, const float* priors) {
  Tree& t = *static_cast<Tree*>(h);
  if (t.status == kLeafSolved) {
    t.k += 1;
    return;
  }
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
  if (t.puct && lh.result == kOpen) {
    const size_t e0 = static_cast<size_t>(node) * t.M;
    const int L = expand(t, node);
    const float uniform = mcts_uniform_prior(L);
    for (int i = 0; i < L; ++i) {
      t.edge_p[e0 + i] = priors != nullptr ? priors[t.edge_action[e0 + i]] : uniform;
      t.edge_key[e0 + i] = mcts_tie_key(t.seed, t.T, static_cast<uint32_t>(node), static_cast<uint32_t>(i));
    }
  }
  if (lh.result != kOpen) {
    if (t.path_node.empty()) {
      t.root_out = mcts_outcome_code(lh, static_cast<int>(lh.ply & 1u));
    } else {
      for (int i = static_cast<int>(t.path_node.size()) - 1; i >= 0; --i) {
        const size_t e0 = static_cast<size_t>(t.path_node[i]) * t.M;
        int mx = 0;
        bool all = true;
        for (int j = 0; j < t.legal[t.path_node[i]]; ++j) {
          mx = t.edge_out[e0 + j] > mx ? t.edge_out[e0 + j] : mx;
          all = all && t.edge_out[e0 + j] != 0;
        }
        const int pv = mcts_proven_value(mx, all);
        if (pv == kUnproven) break;
        if (i > 0)
          t.edge_out[static_cast<size_t>(t.path_node[i - 1]) * t.M + t.path_edge[i - 1]] = mcts_parent_code(pv);
        else
          t.root_out = static_cast<uint8_t>(2 + pv);
      }
    }
  }
  t.k += 1;
}

// Per node slot (creation order): parent slot, action from the parent, N(s), edge count (-1 unexpanded) and
// [slots, M] edge visits / value sums / priors / outcome codes in ascending action order.  Returns the number of
// nodes; *root_code receives the root code, *best the root's BestChild action as mcts_root_stats_kernel<true>.
int sh_dump(void* h, int32_t* node_parent, int32_t* node_action, uint32_t* node_n, int32_t* node_legal,
            uint32_t* edge_n, double* edge_w, float* edge_p, uint8_t* edge_code, int32_t* root_code, int32_t* best) {
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
      edge_code[e] = t.edge_out[e];
    }
  }
  *root_code = t.root_out;
  int bi = -1;
  uint32_t nmax = 0;
  const int L0 = t.legal[0] > 0 ? t.legal[0] : 0;
  for (int i = 0; i < L0; ++i) {
    nmax = t.edge_n[i] > nmax ? t.edge_n[i] : nmax;
    const uint32_t ki = t.puct ? t.edge_key[i] : 0u, kb = (t.puct && bi >= 0) ? t.edge_key[bi] : 0u;
    if (bi < 0 || mcts_puct_best_beats(mcts_outcome_value(t.edge_out[i]), t.edge_n[i], t.edge_w[i], ki, i,
                                       mcts_outcome_value(t.edge_out[bi]), t.edge_n[bi], t.edge_w[bi], kb, bi))
      bi = i;
  }
  // PUCT: -1 while no root edge has a visit; UCT: -1 while the root is terminal or unexpanded
  *best = (bi < 0 || (t.puct && nmax == 0)) ? -1 : t.edge_action[bi];
  return t.nodes;
}

}  // extern "C"
