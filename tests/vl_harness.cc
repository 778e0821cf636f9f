// TEST-ONLY: the search with K leaves per step and virtual loss (mcts_select_kernel / mcts_backup_kernel with
// kVirtual in twixt_mcts.cu) restated for the HOST on the product's helpers (twixt_for_open_spiel_b200/csrc/
// twixt_mcts.cuh: scores, w_eff, draw, tie key, outcome byte, best child, byte formula), the rules
// (twixt_engine.cuh) and the Philox stream, built with -ffp-contract=off, so that `pytest -m "not gpu"` can compare
// it node for node with the executable specification (tests/vl_spec.py) without a GPU.  The storage mirrors the
// device arena: creation-order slots, ascending edges, N / W / child / V per edge and N / V per node, and for a PUCT
// search P / key / outcome per edge.  One call of vh_select_step is one step's K descents; vh_backup_step takes the
// K rows in order.  This file is never part of libtwixt_b200.so.
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

struct Row {
  std::vector<int> path_node, path_edge;
  int leaf = -1;
};

struct Tree {
  int n, rw, M, S, R, K, nodes = 1, k = 0;
  bool puct;
  uint64_t seed;
  uint32_t T;
  double c, vl;
  std::vector<uint32_t> recs;
  std::vector<int32_t> parent, action, legal, child;
  std::vector<uint32_t> node_n, node_v, edge_n, edge_v, edge_key;
  std::vector<uint16_t> edge_action;
  std::vector<double> edge_w;
  std::vector<float> edge_p;
  std::vector<uint8_t> edge_out;
  std::vector<Row> rows;
};

// the ascending legal list of node s, every edge N = 0, W = 0, V = 0, no child (warp_expand)
int expand(Tree& t, int s) {
  const uint32_t* rec = &t.recs[static_cast<size_t>(s) * t.rw];
  const Header h = header_of(rec);
  Rec b{const_cast<uint32_t*>(rec), t.n};
  const size_t e0 = static_cast<size_t>(s) * t.M;
  int L = 0;
  for (int x = 0; x < t.n; ++x) {
    uint32_t w = legal_word(b, h, x);
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
    t.edge_v[e0 + i] = 0;
    t.child[e0 + i] = -1;
  }
  t.legal[s] = L;
  return L;
}

// descent j of the step (simulation k = t.k + j), as select_descents in twixt_mcts.cu
void descend(Tree& t, int j, Row& row) {
  row.path_node.clear();
  row.path_edge.clear();
  int node = 0;
  for (;;) {
    uint32_t* rec = &t.recs[static_cast<size_t>(node) * t.rw];
    const Header hd = header_of(rec);
    if (hd.result != kOpen || t.node_n[node] == 0) break;
    const uint32_t visits_eff = t.node_n[node] + t.node_v[node];
    const size_t e0 = static_cast<size_t>(node) * t.M;
    int edge = -1;
    if (t.puct) {
      const double sq = mcts_sqrt_visits(visits_eff);
      double bs = 0.0;
      uint32_t bk = 0u;
      for (int i = 0; i < t.legal[node]; ++i) {
        const uint8_t o = t.edge_out[e0 + i];
        const uint32_t v = t.edge_v[e0 + i];
        const double sc = o != 0 ? static_cast<double>(mcts_outcome_value(o))
                                 : mcts_puct_score(mcts_virtual_w(t.edge_w[e0 + i], v, t.vl), t.edge_n[e0 + i] + v,
                                                   t.edge_p[e0 + i], sq, t.c);
        if (edge < 0 || mcts_puct_beats(sc, t.edge_key[e0 + i], i, bs, bk, edge)) {
          bs = sc;
          bk = t.edge_key[e0 + i];
          edge = i;
        }
      }
    } else {
      if (t.legal[node] < 0) expand(t, node);
      std::vector<int> unvisited;
      for (int i = 0; i < t.legal[node]; ++i)
        if (t.edge_n[e0 + i] + t.edge_v[e0 + i] == 0u) unvisited.push_back(i);
      if (!unvisited.empty()) {
        edge = unvisited[mcts_draw(t.seed, t.T, static_cast<uint32_t>(t.k + j), static_cast<uint32_t>(unvisited.size()))];
      } else {
        const double log_parent = std::log(static_cast<double>(visits_eff));
        double bs = 0.0;
        for (int i = 0; i < t.legal[node]; ++i) {
          const uint32_t v = t.edge_v[e0 + i];
          const double sc = mcts_uct_score(mcts_virtual_w(t.edge_w[e0 + i], v, t.vl), t.edge_n[e0 + i] + v, log_parent, t.c);
          if (edge < 0 || mcts_score_beats(sc, i, bs, edge)) {
            bs = sc;
            edge = i;
          }
        }
      }
    }
    row.path_node.push_back(node);
    row.path_edge.push_back(edge);
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
      t.legal[ch] = -1;
      t.node_n[ch] = 0;
      t.node_v[ch] = 0;
      t.child[e0 + edge] = ch;
      if (t.puct && chh.result != kOpen) t.edge_out[e0 + edge] = mcts_outcome_code(chh, static_cast<int>(hd.ply & 1u));
    }
    node = t.child[e0 + edge];
  }
  row.leaf = node;
  for (size_t i = 0; i < row.path_node.size(); ++i) {
    t.node_v[row.path_node[i]] += 1;
    t.edge_v[static_cast<size_t>(row.path_node[i]) * t.M + row.path_edge[i]] += 1;
  }
  t.node_v[node] += 1;
}

}  // namespace

extern "C" {

int64_t vh_bytes_per_tree(int n, int max_simulations, int n_rollouts, int puct, int leaves_per_step) {
  const MctsSizes s = mcts_sizes(n, max_simulations, n_rollouts);
  return mcts_parallel_bytes_per_tree(s, puct ? mcts_puct_bytes_per_tree(s) : mcts_bytes_per_tree(s), leaves_per_step);
}

void* vh_create(const uint32_t* root_rec, int n, uint64_t seed, uint32_t tree_stream, int R, double c, int sims,
                int puct, int K, double vl) {
  const MctsSizes s = mcts_sizes(n, sims, R);
  Tree* t = new Tree();
  t->n = n;
  t->rw = static_cast<int>(s.rw);
  t->M = static_cast<int>(s.edges);
  t->S = static_cast<int>(s.slots);
  t->R = R;
  t->K = K;
  t->puct = puct != 0;
  t->seed = seed;
  t->T = tree_stream;
  t->c = c;
  t->vl = vl;
  const size_t S = t->S, E = S * t->M;
  t->recs.assign(S * t->rw, 0u);
  t->parent.assign(S, -1);
  t->action.assign(S, -1);
  t->legal.assign(S, -1);
  t->node_n.assign(S, 0u);
  t->node_v.assign(S, 0u);
  t->child.assign(E, -1);
  t->edge_n.assign(E, 0u);
  t->edge_v.assign(E, 0u);
  t->edge_key.assign(E, 0u);
  t->edge_action.assign(E, 0);
  t->edge_w.assign(E, 0.0);
  t->edge_p.assign(E, 0.0f);
  t->edge_out.assign(E, 0);
  t->rows.resize(K);
  std::memcpy(t->recs.data(), root_rec, t->rw * sizeof(uint32_t));
  return t;
}

void vh_destroy(void* h) { delete static_cast<Tree*>(h); }

// the K descents of one step: leaf records [K, rw], leaf slots [K], statuses [K] (1 = terminal); returns the node
// count
int vh_select_step(void* h, uint32_t* leaves_out, int32_t* leaf_slot, int32_t* status) {
  Tree& t = *static_cast<Tree*>(h);
  for (int j = 0; j < t.K; ++j) {
    descend(t, j, t.rows[j]);
    const uint32_t* lr = &t.recs[static_cast<size_t>(t.rows[j].leaf) * t.rw];
    std::memcpy(leaves_out + static_cast<size_t>(j) * t.rw, lr, t.rw * sizeof(uint32_t));
    leaf_slot[j] = t.rows[j].leaf;
    status[j] = header_of(lr).result != kOpen ? 1 : 0;
  }
  return t.nodes;
}

// rows j = 0 .. K-1 in order: values [K, 2] (nullptr: the mean of R host rollouts on simulation k + j's streams),
// priors [K, n*n] (nullptr: uniform); a PUCT leaf is expanded by the lowest row whose leaf it is
void vh_backup_step(void* h, const float* values, const float* priors) {
  Tree& t = *static_cast<Tree*>(h);
  const int cells = t.n * t.n;
  for (int j = 0; j < t.K; ++j) {
    const Row& row = t.rows[j];
    const int node = row.leaf;
    uint32_t* leaf = &t.recs[static_cast<size_t>(node) * t.rw];
    const Header lh = header_of(leaf);
    double v[2];
    if (lh.result != kOpen) {
      mcts_terminal_value(lh, v);
    } else if (values != nullptr) {
      v[0] = static_cast<double>(values[2 * j]);
      v[1] = static_cast<double>(values[2 * j + 1]);
    } else {
      std::vector<uint32_t> roll(t.rw);
      double s0 = 0.0, s1 = 0.0;
      for (int r = 0; r < t.R; ++r) {
        std::memcpy(roll.data(), leaf, t.rw * sizeof(uint32_t));
        host_playout(roll.data(), t.n, t.seed,
                     mcts_rollout_stream(t.T, static_cast<uint32_t>(t.k), static_cast<uint32_t>(t.R),
                                         static_cast<uint32_t>(r)));
        double ret[2];
        mcts_terminal_value(header_of(roll.data()), ret);
        s0 += ret[0];
        s1 += ret[1];
      }
      v[0] = s0 / t.R;
      v[1] = s1 / t.R;
    }
    for (size_t i = 0; i < row.path_node.size(); ++i) {
      const int p = row.path_node[i];
      const size_t e = static_cast<size_t>(p) * t.M + row.path_edge[i];
      t.node_n[p] += 1;
      t.node_v[p] -= 1;
      t.edge_n[e] += 1;
      t.edge_v[e] -= 1;
      t.edge_w[e] += v[header_of(&t.recs[static_cast<size_t>(p) * t.rw]).ply & 1u];
    }
    t.node_n[node] += 1;
    t.node_v[node] -= 1;
    if (t.puct && lh.result == kOpen && t.legal[node] < 0) {
      const int L = expand(t, node);
      const size_t e0 = static_cast<size_t>(node) * t.M;
      const float uniform = mcts_uniform_prior(L);
      const float* prow = priors != nullptr ? priors + static_cast<size_t>(j) * cells : nullptr;
      for (int i = 0; i < L; ++i) {
        t.edge_p[e0 + i] = prow != nullptr ? prow[t.edge_action[e0 + i]] : uniform;
        t.edge_key[e0 + i] = mcts_tie_key(t.seed, t.T, static_cast<uint32_t>(node), static_cast<uint32_t>(i));
        t.edge_out[e0 + i] = 0;
      }
    }
    t.k += 1;
  }
}

// Per node slot (creation order): parent slot, action from the parent, N(s), V(s), edge count (-1 unexpanded) and
// [slots, M] edge visits / value sums / virtual visits / priors in ascending action order.  Returns the number of
// nodes; *best receives the root's BestChild action as mcts_root_stats_kernel.
int vh_dump(void* h, int32_t* node_parent, int32_t* node_action, uint32_t* node_n, uint32_t* node_v,
            int32_t* node_legal, uint32_t* edge_n, double* edge_w, uint32_t* edge_v, float* edge_p, int32_t* best) {
  Tree& t = *static_cast<Tree*>(h);
  for (int s = 0; s < t.nodes; ++s) {
    node_parent[s] = t.parent[s];
    node_action[s] = t.action[s];
    node_n[s] = t.node_n[s];
    node_v[s] = t.node_v[s];
    node_legal[s] = t.legal[s];
    for (int i = 0; i < (t.legal[s] > 0 ? t.legal[s] : 0); ++i) {
      const size_t e = static_cast<size_t>(s) * t.M + i;
      edge_n[e] = t.edge_n[e];
      edge_w[e] = t.edge_w[e];
      edge_v[e] = t.edge_v[e];
      edge_p[e] = t.edge_p[e];
    }
  }
  int bi = -1;
  uint32_t nmax = 0;
  for (int i = 0; i < (t.legal[0] > 0 ? t.legal[0] : 0); ++i) {
    nmax = t.edge_n[i] > nmax ? t.edge_n[i] : nmax;
    if (t.puct) {
      if (bi < 0 || mcts_puct_best_beats(mcts_outcome_value(t.edge_out[i]), t.edge_n[i], t.edge_w[i], t.edge_key[i], i,
                                         mcts_outcome_value(t.edge_out[bi]), t.edge_n[bi], t.edge_w[bi],
                                         t.edge_key[bi], bi))
        bi = i;
    } else if (bi < 0 || mcts_best_beats(t.edge_n[i], t.edge_w[i], i, t.edge_n[bi], t.edge_w[bi], bi)) {
      bi = i;
    }
  }
  *best = t.puct ? (nmax > 0 ? t.edge_action[bi] : -1) : (bi >= 0 ? t.edge_action[bi] : -1);
  return t.nodes;
}

}  // extern "C"
