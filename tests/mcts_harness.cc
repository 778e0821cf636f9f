// TEST-ONLY: compiles the product's MCTS helpers (twixt_for_open_spiel_b200/csrc/twixt_mcts.cuh) together
// with the rules (twixt_engine.cuh) and the Philox stream (twixt_philox.cuh) for the HOST, built with
// -ffp-contract=off, so that `pytest -m "not gpu"` can run complete searches -- with host-engine rollouts --
// and compare every node with the executable specification (tests/mcts_spec.py) without a GPU.  The node
// storage mirrors the device arena of twixt_mcts.cu (creation-order slots, ascending edges, N / W / child per
// edge); this file is never part of libtwixt_b200.so.
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

// twixt_playout's policy on one record (as tests/host_engine_harness.cc he_playout), played to the end
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

}  // namespace

extern "C" {

double mh_score(double w, uint32_t n, double log_parent, double c) { return mcts_uct_score(w, n, log_parent, c); }

uint32_t mh_draw(uint64_t seed, uint32_t tree_stream, uint32_t k, uint32_t unvisited) {
  return mcts_draw(seed, tree_stream, k, unvisited);
}

int64_t mh_bytes_per_tree(int n, int max_simulations, int n_rollouts) {
  return mcts_bytes_per_tree(mcts_sizes(n, max_simulations, n_rollouts));
}

// One complete search of `sims` simulations from root_rec with R rollouts per leaf.  Outputs per node slot
// (creation order, at most sims + 1): parent slot, action from the parent, N(s), edge count (-1 unexpanded),
// and [slots, M] edge visits / value sums in ascending action order.  Returns the number of nodes; *best
// receives the root's best action (-1 when terminal or unexpanded).
int mh_search(const uint32_t* root_rec, int n, uint64_t seed, uint32_t tree_stream, int R, double c, int sims,
              int32_t* node_parent, int32_t* node_action, uint32_t* node_n, int32_t* node_legal, uint32_t* edge_n,
              double* edge_w, int32_t* best) {
  const MctsSizes s = mcts_sizes(n, sims, R);
  const int rw = static_cast<int>(s.rw), M = static_cast<int>(s.edges), S = static_cast<int>(s.slots);
  std::vector<uint32_t> recs(static_cast<size_t>(S) * rw), roll(rw);
  std::vector<uint16_t> actions(static_cast<size_t>(S) * M);
  std::vector<int32_t> child(static_cast<size_t>(S) * M, -1);
  std::vector<double> logs(S);
  for (int i = 0; i < S; ++i) logs[i] = std::log(static_cast<double>(i));
  std::memcpy(recs.data(), root_rec, rw * sizeof(uint32_t));
  node_parent[0] = -1;
  node_action[0] = -1;
  node_n[0] = 0;
  node_legal[0] = -1;
  int nodes = 1;
  std::vector<int> path_node, path_edge;
  for (int k = 0; k < sims; ++k) {
    path_node.clear();
    path_edge.clear();
    int node = 0;
    for (;;) {
      uint32_t* rec = &recs[static_cast<size_t>(node) * rw];
      const Header h = header_of(rec);
      if (h.result != kOpen || node_n[node] == 0) break;
      const size_t e0 = static_cast<size_t>(node) * M;
      if (node_legal[node] < 0) {
        Rec b{rec, n};
        int L = 0;
        for (int x = 0; x < n; ++x) {
          uint32_t w = legal_word(b, h, x);
          while (w) {
            const int y = tw_ctz(w);
            w &= w - 1u;
            actions[e0 + L] = static_cast<uint16_t>(x * n + y);
            edge_n[e0 + L] = 0;
            edge_w[e0 + L] = 0.0;
            ++L;
          }
        }
        node_legal[node] = L;
      }
      const int L = node_legal[node];
      int unvisited = 0;
      for (int i = 0; i < L; ++i) unvisited += edge_n[e0 + i] == 0 ? 1 : 0;
      int edge = -1;
      if (unvisited > 0) {
        int j = static_cast<int>(mcts_draw(seed, tree_stream, static_cast<uint32_t>(k), static_cast<uint32_t>(unvisited)));
        for (int i = 0; i < L && edge < 0; ++i)
          if (edge_n[e0 + i] == 0 && j-- == 0) edge = i;
      } else {
        double bs = 0.0;
        for (int i = 0; i < L; ++i) {
          const double sc = mcts_uct_score(edge_w[e0 + i], edge_n[e0 + i], logs[node_n[node]], c);
          if (edge < 0 || mcts_score_beats(sc, i, bs, edge)) {
            bs = sc;
            edge = i;
          }
        }
      }
      path_node.push_back(node);
      path_edge.push_back(edge);
      if (child[e0 + edge] < 0) {
        const int ch = nodes++;
        uint32_t* crec = &recs[static_cast<size_t>(ch) * rw];
        std::memcpy(crec, rec, rw * sizeof(uint32_t));
        Rec cb{crec, n};
        Header chh = h;
        const int a = actions[e0 + edge];
        apply_legal_cell<kStack>(cb, chh, a / n, a % n);
        store_header(cb, chh);
        node_parent[ch] = node;
        node_action[ch] = a;
        node_n[ch] = 0;
        node_legal[ch] = -1;
        child[e0 + edge] = ch;
      }
      node = child[e0 + edge];
    }
    const uint32_t* leaf = &recs[static_cast<size_t>(node) * rw];
    const Header lh = header_of(leaf);
    double v[2];
    if (lh.result != kOpen) {
      mcts_terminal_value(lh, v);
    } else {
      double s0 = 0.0, s1 = 0.0;
      for (int r = 0; r < R; ++r) {
        std::memcpy(roll.data(), leaf, rw * sizeof(uint32_t));
        host_playout(roll.data(), n, seed, mcts_rollout_stream(tree_stream, static_cast<uint32_t>(k), R, r));
        double ret[2];
        mcts_terminal_value(header_of(roll.data()), ret);
        s0 += ret[0];
        s1 += ret[1];
      }
      v[0] = s0 / R;
      v[1] = s1 / R;
    }
    for (size_t i = 0; i < path_node.size(); ++i) {
      const int p = path_node[i];
      const size_t e = static_cast<size_t>(p) * M + path_edge[i];
      node_n[p] += 1;
      edge_n[e] += 1;
      edge_w[e] += v[header_of(&recs[static_cast<size_t>(p) * rw]).ply & 1u];
    }
    node_n[node] += 1;
  }
  int bi = -1;
  for (int i = 0; i < (node_legal[0] > 0 ? node_legal[0] : 0); ++i)
    if (bi < 0 || mcts_best_beats(edge_n[i], edge_w[i], i, edge_n[bi], edge_w[bi], bi)) bi = i;
  *best = bi < 0 ? -1 : actions[bi];
  return nodes;
}

}  // extern "C"
