// twixt_kernels.cuh -- launch wrappers of the sm_100a kernels (defined in
// twixt_kernels_api.cu and twixt_kernel_playout.cu).  All env state is an
// array of records in global memory: records + env * record_words(n).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/twixt_b200.h"

namespace twixt {

// device-side counters, one per batch (twixt_stats in the C ABI)
struct DeviceStats {
  unsigned long long plies;
  unsigned long long games;
  unsigned long long red_wins;
  unsigned long long blue_wins;
  unsigned long long draws;
  unsigned long long swaps;
  unsigned long long max_length;
  // lowest index (within the call's range) of an illegal action seen by the
  // apply kernel, 0xFFFFFFFF = none
  unsigned int illegal_index;
  unsigned int pad;
  // ticket counter of the persistent playout kernel (zeroed before every launch)
  unsigned long long tickets;
  // validate kernel: (lowest invalid env << 8) | reason, all ones = every record passed
  unsigned long long invalid_code;
  // replay kernel: (lowest env that met an illegal action << 32) | that action, all ones = none
  unsigned long long replay_illegal;
  // clone kernel: lowest position whose gathered source id was out of range / inside the destination
  unsigned int bad_clone_index;
  unsigned int pad2;
  // only written by the bounds-instrumented test variant of the playout kernel (TW_PLAYOUT_BOUNDS_CHECK)
  unsigned long long bounds_violations;
};

struct PlayoutArgs {
  uint32_t* records;           // first env of the range
  int64_t count;
  int n;
  int max_plies;
  uint64_t seed;
  uint64_t stream_base;        // stream id of range element 0 when stream_ids == nullptr
  const uint64_t* stream_ids;  // [count] or nullptr
  float* out_returns;          // [count,2] or nullptr
  int32_t* out_lengths;        // [count] or nullptr
  uint16_t* out_actions;       // [trace_plies, count] or nullptr
  int trace_plies;
  DeviceStats* stats;
  unsigned long long* tickets;  // &stats->tickets
};

// Device arena of a batched MCTS search (twixt_mcts.cu; sizes and byte formula in twixt_mcts.cuh).  Tree t owns
// node slots [t*S, (t+1)*S) (slot 0 of a tree is its root), path entries [t*P, (t+1)*P) and rollout slots
// [t*R, (t+1)*R); the edges of global node slot g are [g*M, (g+1)*M).
struct MctsArena {
  int n, rw, M, S, P, R;
  uint32_t* node_rec;       // [trees*S*rw] state record of each node
  int32_t* node_legal;      // [trees*S] number of edges, -1 while the node is not expanded
  uint32_t* node_n;         // [trees*S] N(s)
  uint16_t* edge_action;    // [trees*S*M] ascending legal actions
  uint32_t* edge_n;         // [trees*S*M] N(a)
  double* edge_w;           // [trees*S*M] W(a)
  int32_t* edge_child;      // [trees*S*M] child slot within the tree, -1 = none yet
  int4* tree;               // [trees] node count, leaf slot, path length, leaf status
  int2* path;               // [trees*P] (node slot, edge << 1 | player to move at that node)
  uint32_t* roll_rec;       // [trees*R*rw] rollout slots
  uint64_t* roll_ids;       // [trees*R] their Philox stream ids
  float* roll_ret;          // [trees*R*2] their returns
  const double* log_table;  // [S] log(i)
  // PUCT searches only (nullptr in a UCT search, which selects on that)
  float* edge_p;            // [trees*S*M] prior P(a), written when the node is expanded at its backup
  uint32_t* edge_key;       // [trees*S*M] tie key (mcts_tie_key)
  uint8_t* edge_out;        // [trees*S*M] terminal outcome of the child (mcts_outcome_code), 0 = none; a solver
                            // search (UCT ones too) also writes the code of a proven child here
  // solver searches only (nullptr otherwise, which selects on that)
  uint8_t* root_out;        // [trees] outcome code of the root (twixt_mcts.cuh), 0 = unproven; cleared by begin
  // searches with K > 1 leaves per step only (nullptr otherwise, which selects on that).  Their tree entries, paths
  // and rollout slots are per leaf row t*K + j: tree [trees*K], path [trees*K*P], rollout slots [trees*K*R]; the
  // node count of tree t is in tree[t*K].x
  uint16_t* node_v;         // [trees*S] virtual visits V(s), 0 between steps
  uint16_t* edge_v;         // [trees*S*M] virtual visits V(a), 0 between steps
  int K;                    // leaves per step (1 without node_v)
  double vl;                // virtual loss
};

cudaError_t launch_mcts_begin(const MctsArena& a, const uint32_t* roots, int64_t count, cudaStream_t s);
// leaf_dst == nullptr: leaves go to the rollout slots (built-in evaluator), else to records leaf_dst + t*rw
cudaError_t launch_mcts_select(const MctsArena& a, int64_t count, uint64_t seed, uint32_t stream0, uint32_t k,
                               double uct_c, uint32_t* leaf_dst, int32_t* out_status, cudaStream_t s);
// values == nullptr: the mean of the R rollout returns, else the caller's [count, 2] float32.  A PUCT search
// expands each non-terminal leaf with priors [count, n*n] float32 (nullptr: uniform over the legal actions).
cudaError_t launch_mcts_backup(const MctsArena& a, int64_t count, const float* values, const float* priors,
                               uint64_t seed, uint32_t stream0, cudaStream_t s);
cudaError_t launch_mcts_root_stats(const MctsArena& a, int64_t count, int32_t* out_visits, double* out_value_sums,
                                   int32_t* out_best, cudaStream_t s);
// solver searches: proven [count] u8, returns [count, 2] f32, edge values [count, n*n] i8, N(root) [count] i32
cudaError_t launch_mcts_solver_stats(const MctsArena& a, int64_t count, uint8_t* out_proven, float* out_returns,
                                     int8_t* out_edge_values, int32_t* out_simulations, cudaStream_t s);
// tree reuse: actions [count] (device), map [count*S] int32 scratch, out_status [count] or nullptr; an illegal action
// lowers *illegal_index to its tree
cudaError_t launch_mcts_advance(const MctsArena& a, int64_t count, const int32_t* actions, int keep_nodes,
                                int32_t* map, int32_t* out_status, unsigned int* illegal_index, cudaStream_t s);
// PUCT searches: P(a) of the root edges of every expanded root from priors [count, n*n] (device)
cudaError_t launch_mcts_set_root_priors(const MctsArena& a, int64_t count, const float* priors, cudaStream_t s);

cudaError_t launch_reset(uint32_t* records, int64_t count, int n, cudaStream_t s);
cudaError_t launch_clone(uint32_t* dst, const uint32_t* src, const int64_t* src_ids, int64_t count, int n,
                         int64_t num_envs, int64_t dst_first, DeviceStats* stats, cudaStream_t s);
cudaError_t launch_replay(uint32_t* records, int64_t count, int n, const int32_t* actions, int64_t stride,
                          const int32_t* lengths, int32_t* out_applied, DeviceStats* stats, cudaStream_t s);
cudaError_t launch_step(uint32_t* record, int n, int action, twixt_step_result* out, int64_t* out_legal, cudaStream_t s);
cudaError_t launch_validate(const uint32_t* records, int64_t count, int n, DeviceStats* stats, cudaStream_t s);
const char* invalid_reason_text(unsigned code);
cudaError_t launch_legal_actions(const uint32_t* records, int64_t count, int n, void* out_actions, int elem_bytes,
                                 int64_t stride, int32_t* out_counts, cudaStream_t s);
cudaError_t launch_legal_mask(const uint32_t* records, int64_t count, int n, uint8_t* out, cudaStream_t s);
cudaError_t launch_apply(uint32_t* records, int64_t count, int n, const int32_t* actions, int32_t* out_status,
                         DeviceStats* stats, cudaStream_t s);
cudaError_t launch_query(const uint32_t* records, int64_t count, int n, int8_t* out_player, uint8_t* out_terminal,
                         float* out_returns, cudaStream_t s);
cudaError_t launch_observation(const uint32_t* records, int64_t count, int n, float* out, uint8_t* out_mask,
                               cudaStream_t s);
cudaError_t launch_playout(const PlayoutArgs& a, cudaStream_t s);
// one-time per-process setup of the playout kernels (opt-in shared memory)
cudaError_t playout_setup();
// the five size groups of twixt_kernel_playout.cu (board sizes 5+g, 10+g, 15+g, 20+g)
cudaError_t playout_setup_g0();
cudaError_t playout_setup_g1();
cudaError_t playout_setup_g2();
cudaError_t playout_setup_g3();
cudaError_t playout_setup_g4();
cudaError_t launch_playout_g0(const PlayoutArgs& a, cudaStream_t s);
cudaError_t launch_playout_g1(const PlayoutArgs& a, cudaStream_t s);
cudaError_t launch_playout_g2(const PlayoutArgs& a, cudaStream_t s);
cudaError_t launch_playout_g3(const PlayoutArgs& a, cudaStream_t s);
cudaError_t launch_playout_g4(const PlayoutArgs& a, cudaStream_t s);

}  // namespace twixt
