/* twixt_b200.h -- C ABI of libtwixt_b200.so, the B200-native batched TwixT engine.
 *
 * This is the drop-in boundary for the hot path of
 * stevens68/TwixT_for_open_spiel: one batched entry point per method of the
 * open_spiel Game/State surface that the reference overrides in
 *   open_spiel/games/twixt/twixt.h:31-146  and  twixt.cc:35-145.
 * A binding for open_spiel (C++), pyspiel-style Python (ctypes) or any other
 * FFI only needs this header; no CUDA, torch or C++ types appear in it.
 *
 * Conventions
 *  - Every call returns TWIXT_OK (0) or a negative TWIXT_E* code and never
 *    aborts the process (the reference calls SpielFatalError, twixt.h:96,
 *    twixt.cc:140-143).  twixt_last_error() returns the message of the last
 *    failing call on the calling thread; messages that the reference pins are
 *    reproduced byte for byte ("board_size out of range [5..24]: 30",
 *    "Not a legal action: 11").
 *  - A batch holds `num_envs` independent games ("envs") of one board size in
 *    device memory.  Batched calls address the contiguous env range
 *    [first, first+count).
 *  - Every data pointer may be a DEVICE pointer (cudaMalloc / torch CUDA
 *    tensor: the kernel reads/writes it directly, asynchronously on the
 *    batch's stream) or a HOST pointer (pageable or pinned: the library stages
 *    it -- small transfers through a pinned, device-mapped arena the kernel
 *    accesses directly, large ones through device scratch -- and the call
 *    returns after the data arrived).  The kind is detected with
 *    cudaPointerGetAttributes.
 *  - A batch is not thread-safe; distinct batches are independent.
 *  - There is no CPU fallback: every entry point that touches game state
 *    launches sm_100a kernels and fails with TWIXT_ECUDA when no such device
 *    is present.
 *
 * State record (what twixt_export_state / twixt_import_state move, and what
 * lives in HBM): per env `record_words` 32-bit words, 16-byte aligned:
 *    word 0  ply            (Board::move_counter_, twixtboard.h:75)
 *    word 1  bits 0-1 result (0 open 1 red won 2 blue won 3 draw, twixtboard.h:48)
 *            bit 2 swapped   (twixtboard.h:76)
 *    word 2  action of the first move (Board::move_one_), 0xFFFFFFFF before it
 *    word 3  bits 0-15 / 16-31: number of empty cells red / blue may play on
 *    then 9 bit-planes of n column words each; bit y of word x <=> cell (x,y),
 *    x = column, y = row counted from the bottom (twixtboard.h:153-213):
 *      0 red pegs                 1 blue pegs
 *      2..5 links NNE, ENE, ESE, SSE stored at their WEST endpoint
 *            (Cell::links_ bits 0..3 there, bits 4..7 at the other end,
 *             twixtcell.h:58-78)
 *      6 / 7 peg is linked to its owner's start / end border line
 *            (Cell::linked_to_border_, twixtcell.h:89-95,107)
 *      8 peg has a blocked neighbour in an east direction
 *            (Cell::HasBlockedNeighborsEast, twixtcell.h:82-84)
 *    zero padding up to a multiple of 4 words.
 */
#ifndef TWIXT_B200_H_
#define TWIXT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TWIXT_MIN_BOARD_SIZE 5      /* twixtboard.h:32 */
#define TWIXT_MAX_BOARD_SIZE 24     /* twixtboard.h:33 */
#define TWIXT_DEFAULT_BOARD_SIZE 8  /* twixtboard.h:34 */
#define TWIXT_NUM_OBS_PLANES 12     /* twixtboard.h:46 */
#define TWIXT_TERMINAL_PLAYER (-4)  /* open_spiel kTerminalPlayerId, playthrough.txt:678 */
#define TWIXT_HEADER_WORDS 4
#define TWIXT_NUM_STATE_PLANES 9

enum {
  TWIXT_OK = 0,
  TWIXT_EINVAL = -1,   /* bad argument (range, null pointer, size) */
  TWIXT_ECUDA = -2,    /* CUDA runtime error / no sm_100 device */
  TWIXT_EILLEGAL = -3, /* twixt_apply: at least one action was not legal */
  TWIXT_ENOMEM = -4
};

typedef struct twixt_batch twixt_batch;

/* Game-level constants.  Mirrors TwixTGame's accessors, twixt.h:122-141. */
typedef struct twixt_game_info {
  int32_t board_size;
  int32_t num_distinct_actions; /* n*n            twixt.h:122-124 */
  int32_t num_players;          /* 2              twixt.h:126 */
  int32_t max_game_length;      /* n*n-4+1        twixt.h:136-139 */
  int32_t obs_shape[3];         /* {12, n, n-2}   twixt.h:131-134 (without its static-shape bug) */
  int32_t obs_size;             /* 12*n*(n-2) */
  int32_t max_legal_actions;    /* n*(n-2)        twixtboard.cc:253 */
  int32_t record_words;         /* words per env state record */
  double min_utility;           /* -1  twixt.h:127 */
  double max_utility;           /* +1  twixt.h:129 */
  double utility_sum;           /*  0  twixt.h:128 */
} twixt_game_info;

/* Aggregate counters of the playouts run on a batch since the last
 * twixt_stats_reset (the only quantity ever reduced across GPUs). */
typedef struct twixt_stats {
  int64_t plies;      /* moves applied inside twixt_playout */
  int64_t games;      /* envs that reached a terminal state inside twixt_playout */
  int64_t red_wins;
  int64_t blue_wins;
  int64_t draws;
  int64_t swaps;      /* playouts in which the swap rule was used */
  int64_t max_length; /* longest finished game (plies) */
  int64_t kernel_launches; /* kernels launched by this batch since creation */
  int64_t debug_violations; /* always 0 in the product build; the bounds-instrumented test variant of the
                               playout kernel counts accesses outside an env's own storage here */
} twixt_stats;

const char* twixt_last_error(void);
const char* twixt_version(void);

/* TwixTGame::TwixTGame range check, twixt.cc:134-145.  No GPU needed. */
int twixt_game_info_for(int board_size, twixt_game_info* out);

/* Replaces TwixTGame construction + NewInitialState() (twixt.h:118-120,
 * twixt.cc:62-65) for num_envs games at once: allocates the records on
 * `device` and resets every env to the initial position.  `seed` keys the
 * Philox streams of twixt_playout. */
int twixt_create(int board_size, int64_t num_envs, int device, uint64_t seed, twixt_batch** out);
void twixt_destroy(twixt_batch* b);
int twixt_get_info(const twixt_batch* b, twixt_game_info* out);
int64_t twixt_num_envs(const twixt_batch* b);

/* Use an existing CUDA stream (e.g. torch's current stream) instead of the
 * batch's own; pass the cudaStream_t as an integer. */
int twixt_set_stream(twixt_batch* b, uintptr_t cuda_stream);
uintptr_t twixt_get_stream(const twixt_batch* b);
int twixt_synchronize(twixt_batch* b);
int twixt_set_seed(twixt_batch* b, uint64_t seed);
/* Philox stream id of env 0 of this batch when twixt_playout gets no
 * stream_ids (env i uses base + i): lets shards on several GPUs draw from
 * disjoint streams so results do not depend on the GPU count. */
int twixt_set_stream_base(twixt_batch* b, uint64_t base);

/* NewInitialState(), twixt.h:118-120 / Board::Board twixtboard.cc:168-174. */
int twixt_reset(twixt_batch* b, int64_t first, int64_t count);

/* State::Clone(), twixt.h:80-82.  dst env i <- src env i (ranges may not
 * overlap), or dst env first+i <- env src_ids[i] for the gather form
 * (src_ids: int64, host or device).  Every id must lie in [0, num_envs) and outside the destination range;
 * an offending id copies nothing for its env and fails the call with TWIXT_EINVAL (ids on the device are
 * checked by the kernel itself).  twixt_clone_from rejects overlapping ranges within one batch. */
int twixt_clone(twixt_batch* b, int64_t src_first, int64_t dst_first, int64_t count);
int twixt_clone_gather(twixt_batch* b, const int64_t* src_ids, int64_t dst_first, int64_t count);
/* Clone between two batches of the same board size (possibly on one device). */
int twixt_clone_from(twixt_batch* dst, int64_t dst_first, const twixt_batch* src, int64_t src_first,
                     int64_t count);

/* TwixTState::LegalActions(), twixt.h:86-90: ascending actions of the player
 * to move, empty when terminal.  out_actions is [count, stride] with
 * stride >= max_legal_actions elements of elem_bytes (2: uint16, 4: int32,
 * 8: int64 = open_spiel::Action); entries past the count are left untouched.
 * out_counts is [count] int32.  Either pointer may be null. */
int twixt_legal_actions(twixt_batch* b, int64_t first, int64_t count, void* out_actions,
                        int32_t elem_bytes, int64_t stride, int32_t* out_counts);

/* Upstream State::LegalActionsMask(): [count, n*n] uint8, 1 = legal. */
int twixt_legal_mask(twixt_batch* b, int64_t first, int64_t count, uint8_t* out_mask);

/* State::ApplyAction -> TwixTState::DoApplyAction, twixt.h:93-104 ->
 * Board::ApplyAction, twixtboard.cc:457-499.  actions is [count] int32, one
 * per env; a negative action skips that env.  out_status (nullable) is
 * [count] int32: 0 applied, 1 "Not a legal action" (env left unchanged),
 * 2 skipped.  Returns TWIXT_EILLEGAL if any env reported 1 (only checked when
 * out_status is a host pointer or null); the message names the first such
 * action like the reference does. */
int twixt_apply(twixt_batch* b, int64_t first, int64_t count, const int32_t* actions,
                int32_t* out_status);

/* CurrentPlayer() twixt.h:38 (0 red, 1 blue, -4 terminal), IsTerminal()
 * twixt.h:45-48, Returns() twixt.h:50-63 ([count,2] float32: +-1 or 0). */
int twixt_current_player(twixt_batch* b, int64_t first, int64_t count, int8_t* out);
int twixt_is_terminal(twixt_batch* b, int64_t first, int64_t count, uint8_t* out);
int twixt_returns(twixt_batch* b, int64_t first, int64_t count, float* out);

/* TwixTState::ObservationTensor, twixt.cc:76-132: [count, 12, n, n-2]
 * float32, zero-filled then 1.0s; identical for both players. */
int twixt_observation(twixt_batch* b, int64_t first, int64_t count, float* out);

/* ObservationTensor + LegalActionsMask of the same envs in ONE pass over the records (the producer of an
 * AlphaZero-style inference batch, BASELINE config C5): out_obs as twixt_observation, out_mask as
 * twixt_legal_mask; bit-identical to the two separate calls. */
int twixt_observation_and_mask(twixt_batch* b, int64_t first, int64_t count, float* out_obs,
                               uint8_t* out_mask);

/* Replays a whole action history per env in one launch: upstream serialises a state as its action history
 * (State::Serialize) and Game::DeserializeState re-applies it move by move; the reference has no UndoAction
 * (twixt.h:84), so replay is also how a search returns to an earlier position.  actions is [count, stride]
 * int32; env first+i applies actions[i*stride + k] for k = 0 .. len_i-1 from its CURRENT state, with the
 * legality test of DoApplyAction (twixt.h:93-104) before every move, where len_i = lengths[i] (nullable:
 * then a row ends at its first negative entry or at stride).  An env stops at its first illegal action,
 * keeping the state reached; out_applied (nullable) is [count] int32 = moves made.  Returns TWIXT_EILLEGAL
 * with the reference's message for the lowest such env (only checked when out_applied is null or any
 * pointer is a host pointer; with device pointers throughout the call is asynchronous). */
int twixt_replay(twixt_batch* b, int64_t first, int64_t count, const int32_t* actions, int64_t stride,
                 const int32_t* lengths, int32_t* out_applied);

/* One State step for an UNBATCHED caller -- what upstream example.cc / mcts_example.cc do per move:
 * ApplyAction, then IsTerminal / CurrentPlayer / Returns / LegalActions of the new state (twixt.h:38-104).
 * One kernel launch does all of it for env `env`: `action` >= 0 is applied with the legality test of
 * DoApplyAction (status 1 and TWIXT_EILLEGAL "Not a legal action: N" if illegal, env unchanged),
 * TWIXT_STEP_QUERY applies nothing, TWIXT_STEP_RESET resets the env to the initial position first; then
 * `out` and the ascending `out_legal` ([max_legal_actions] int64 = open_spiel::Action, nullable) describe the
 * resulting state.  An adapter keeps the answer with its State object, so the four query methods cost no
 * further GPU call until the next ApplyAction (twixt_for_open_spiel_b200/adapter). */
#define TWIXT_STEP_QUERY (-1)
#define TWIXT_STEP_RESET (-2)
typedef struct twixt_step_result {
  int32_t status;         /* 0 applied / nothing to apply, 1 illegal action */
  int32_t current_player; /* 0, 1 or TWIXT_TERMINAL_PLAYER */
  int32_t is_terminal;
  int32_t num_legal;      /* entries written to out_legal (0 when terminal) */
  float returns[2];
} twixt_step_result;
int twixt_step(twixt_batch* b, int64_t env, int32_t action, twixt_step_result* out, int64_t* out_legal);

/* The random-playout loop of upstream example.cc / RandomRolloutEvaluator
 * (LegalActions -> uniform pick -> ApplyAction until IsTerminal), fused into
 * one kernel with the env state held on chip.  Every env in the range is
 * played from its CURRENT state until it is terminal or max_plies moves were
 * made, and is left in the state reached.  Move `step` (0-based within this
 * call) of an env picks index (word*L)>>32 of its ascending legal list of
 * length L, where word = Philox4x32-10(key=seed, counter=(stream, step>>2,0))
 * [step&3] and stream = stream_ids[i] if given, else the env index.
 * Outputs (all nullable): out_returns [count,2] float32, out_lengths [count]
 * int32 = moves made by THIS call, out_actions [max_plies_traced, count]
 * uint16 step-major action trace (0xFFFF where no move was made) with
 * trace_plies rows. */
int twixt_playout(twixt_batch* b, int64_t first, int64_t count, int32_t max_plies,
                  const uint64_t* stream_ids, float* out_returns, int32_t* out_lengths,
                  uint16_t* out_actions, int32_t trace_plies);

/* Raw state records, [count, record_words] uint32 (host or device).
 * The reference can only reach a state through DoApplyAction (twixt.h:93-104); records handed to
 * twixt_import_state are therefore VALIDATED on the device before any env is overwritten (header ranges,
 * peg placement and counts, link endpoints, flag/blocked bits on pegs only, recounted legal-cell counters,
 * zero padding).  A bad record fails the whole call with TWIXT_EINVAL, "invalid state record at index I:
 * <reason>", and leaves the batch untouched.  twixt_set_validation(b, 0) skips the check for trusted
 * records (a plain copy, asynchronous for device pointers); the default is on. */
int twixt_export_state(twixt_batch* b, int64_t first, int64_t count, uint32_t* out_records);
int twixt_import_state(twixt_batch* b, int64_t first, int64_t count, const uint32_t* records);
int twixt_set_validation(twixt_batch* b, int enabled);

int twixt_get_stats(twixt_batch* b, twixt_stats* out);
int twixt_stats_reset(twixt_batch* b);

/* Batched MCTS: `num_trees` independent searches on the device, each open_spiel's MCTSBot with
 * RandomRolloutEvaluator(n_rollouts), solve = false (the solver is TWIXT_MCTS_SOLVE, below) and no Dirichlet
 * noise, made deterministic:
 *  - twixt_mcts_begin: the root of tree t is a COPY of env root_first + t (later changes to that env do not
 *    affect the tree); its stream id is T = stream_base + root_first + t (twixt_set_stream_base, so results do
 *    not depend on sharding), which must be below 2^32.  The batch's seed at begin keys every draw.
 *  - simulation k (k = 0, 1, .. since begin) descends from the root: it stops at a terminal node or at a node
 *    with N(s) == 0 (the leaf); a node is expanded on its second visit (one edge per legal action, ascending,
 *    the swap offer included at ply 1); if U > 0 edges are unvisited it takes the j-th of them in ascending
 *    order, j = (w*U) >> 32 with w = word 0 of Philox4x32-10(key = seed, counter = (T lo, T hi, k, 1)), and
 *    creates its child; otherwise it takes the edge of largest W/N + c*sqrt(ln N(s) / N) (IEEE double, no
 *    contraction, ln from the host's libm; ties to the lowest action).
 *  - the leaf value v: Returns() for a terminal leaf; else the mean of R fused playouts from the leaf
 *    (rollout r on stream (T << 32) | (k*R + r), as twixt_playout), or in the stepwise form the caller's
 *    float value.  Every node on the path gets N += 1, every edge N += 1 and W += v[player to move at its
 *    parent].
 * twixt_mcts_run(k) queues k simulations (three kernel launches each: select, playout, backup; no host
 * synchronisation).  Stepwise form: twixt_mcts_select writes each tree's leaf record into batch envs
 * [leaf_first, leaf_first + count) and out_leaf_status [count] int32 (nullable: 0 needs a value, 1 terminal:
 * its value is Returns()); the caller evaluates them (e.g. twixt_observation_and_mask + a value network) and
 * hands twixt_mcts_backup [count, 2] float32 values (entries of terminal leaves are ignored).  run and the
 * stepwise pair share the same kernels and may be mixed.  twixt_mcts_root_stats: out_visits [count, n*n]
 * int32 and out_value_sums [count, n*n] double are N(a) / W(a) of the root edges (0 for other actions),
 * out_best [count] int32 is open_spiel's BestChild (most visits, then larger W, then lowest action), -1 while
 * the root is terminal or unexpanded; each pointer is nullable.
 * Errors (TWIXT_EINVAL, trees unchanged): ranges outside the batch, count > num_trees, more than
 * max_simulations simulations since begin, select twice in a row, backup without select, run while a select
 * is pending, uct_c not finite or negative, stream ids out of range (T >= 2^32, max_simulations *
 * n_rollouts >= 2^32).  twixt_mcts_create computes the arena size (per tree: (max_simulations + 1) node slots
 * of record + 18 bytes per legal action, twixt_mcts.cuh) and fails with TWIXT_ENOMEM, naming it, when the
 * device has less free memory.  The rollouts count in the batch's twixt_stats like any twixt_playout call.
 * A search uses its batch's stream and must be destroyed before the batch. */
typedef struct twixt_mcts twixt_mcts;
int twixt_mcts_create(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                      double uct_c, twixt_mcts** out);
void twixt_mcts_destroy(twixt_mcts* m);
int twixt_mcts_begin(twixt_mcts* m, int64_t root_first, int64_t count);
int twixt_mcts_run(twixt_mcts* m, int32_t num_simulations);
int twixt_mcts_select(twixt_mcts* m, int64_t leaf_first, int32_t* out_leaf_status);
int twixt_mcts_backup(twixt_mcts* m, const float* values);
int twixt_mcts_root_stats(twixt_mcts* m, int32_t* out_visits, double* out_value_sums, int32_t* out_best);

/* PUCT search with policy priors (AlphaZero): open_spiel's MCTSBot with child_selection_fn = puct_value and
 * solve = false (open_spiel python/algorithms/mcts.py: SearchNode.puct_value, SearchNode.sort_key,
 * _apply_tree_policy, mcts_search), made deterministic.  As above: the root is a copy of an env, the tree
 * stream id is T, a simulation descends until a terminal node or a node with N(s) == 0, the backup adds
 * v[player to move at the parent] to every edge on the path, nodes are numbered in creation order.  What differs:
 *  - every edge carries a prior P(a) (float32).  A non-terminal leaf is EXPANDED AT ITS BACKUP: one edge per
 *    legal action, ascending (swap offer at ply 1), N = 0, W = 0, P(a) = priors[t, a] from the caller
 *    (open_spiel expands on the second visit from evaluator.prior, which AlphaZeroEvaluator answers from the
 *    network call that valued the leaf).  Without priors (twixt_mcts_run, twixt_mcts_backup, or a null
 *    pointer) P(a) = float32(1.0 / L), RandomRolloutEvaluator.prior.  Prior entries of illegal actions, and all
 *    entries of terminal leaves, are ignored.
 *  - edge a under node s scores, in IEEE double without contraction, q = N(a) > 0 ? W(a)/N(a) : 0,
 *    u = ((c * (double)P(a)) * sqrt((double)N(s))) / (double)(N(a) + 1), q + u.  Unvisited edges are scored
 *    like any other (there is no unvisited-edge draw).  An edge whose child exists and is terminal scores
 *    Returns()[player to move at s] (-1, 0 or +1), with no exploration term.
 *  - ties reproduce open_spiel's shuffle of the children at expansion: edge i of node slot s has the tie key
 *    word 0 of Philox4x32-10(key = seed, counter = (T, s, i, 2)); among equal scores the smaller key wins,
 *    then the lower edge.
 *  - out_best of twixt_mcts_root_stats is sort_key's maximum: (terminal child ? Returns()[root player] : 0),
 *    then N(a), then W(a), then the tie rule; -1 while every root edge has N = 0.
 *  - Dirichlet noise is the caller's: simulation 0's leaf is always the root, so mixing (1-eps)*p +
 *    eps*Dir(alpha) over each row's legal actions into the priors of the FIRST backup after begin gives
 *    open_spiel's root noise (mcts.py add_dirichlet_noise does this in float32, where open_spiel mixes in
 *    double).
 * twixt_mcts_backup_priors: priors [count, n*n] float32 on the host or the device, or NULL (= twixt_mcts_backup).
 * Host priors must be finite and >= 0 everywhere, else TWIXT_EINVAL before anything is launched (trees
 * unchanged); device priors are the caller's responsibility (no input makes the search take an edge outside
 * the node's legal list).  Priors given to a UCT search: TWIXT_EINVAL.  run, select, backup, root_stats and
 * destroy work on both kinds with the same errors and launch counts.  The arena adds 9 bytes per edge (prior,
 * tie key, outcome byte; twixt_mcts.cuh). */
int twixt_mcts_create_puct(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                           double uct_c, twixt_mcts** out);
int twixt_mcts_backup_priors(twixt_mcts* m, const float* values, const float* priors);

/* MCTS-Solver (open_spiel MCTSBot(..., solve=True), its default; python/algorithms/mcts.py mcts_search).
 * twixt_mcts_create_ex takes flags: TWIXT_MCTS_PUCT selects PUCT (flags 0 and TWIXT_MCTS_PUCT are exactly
 * twixt_mcts_create and twixt_mcts_create_puct), TWIXT_MCTS_SOLVE adds the solver to either kind; other bits are
 * TWIXT_EINVAL.  Everything above holds, plus:
 *  - every edge has an outcome code: 0 unknown, else 2 + the child's value for the player to move at the parent
 *    (1 loss, 2 draw, 3 win).  It is set when a terminal child is created and when a child becomes proven.
 *  - proof pass: in the backup of a simulation whose leaf is terminal, and only then, walking up the path from
 *    the leaf's parent: node c (player to move p) is proven when some edge of c has code 3 (a win for p) or
 *    all of its edges have non-zero codes; its value is v = max(code) - 2 and the parent's edge into c gets
 *    code 2 - v (zero-sum, players alternate by ply: the swap is blue's move at ply 1).  The walk stops at the
 *    first node that is not proven.  A proven root, or a terminal root at its first simulation (with
 *    Returns()), makes the tree FINISHED.
 *  - a finished tree does nothing in later simulations: select takes no path and reports leaf status 2
 *    (TWIXT_MCTS_LEAF_SOLVED), the stepwise form leaves env leaf_first + t untouched, backup ignores that
 *    row's values and priors, and its rollout slots add no plies and no games to twixt_stats.  The
 *    simulation counter and the max_simulations check do not change.
 *  - UCT + solve: a visited edge with a non-zero code scores its value (-1, 0, +1) instead of the UCT term
 *    (open_spiel uct_value); the unvisited-edge draw comes first as before.  out_best of twixt_mcts_root_stats is
 *    open_spiel's sort_key: (outcome value, N, W), then the lowest action; -1 while the root is terminal or
 *    unexpanded.  PUCT + solve: selection and out_best read the codes as PUCT does for terminal children.
 *  - arena: 1 byte per tree more, and a UCT search 1 byte per edge (twixt_mcts.cuh).
 * twixt_mcts_solver_stats: out_proven [count] u8 (1 once the root is proven), out_returns [count, 2] float32
 * (open_spiel's root.outcome: Returns() of the proven result, (0, 0) while unproven), out_edge_values
 * [count, n*n] int8 (-1, 0 or +1 for a proven root move, from the view of the player to move at the root;
 * TWIXT_MCTS_UNPROVEN elsewhere), out_simulations [count] int32 (N(root): the simulations the tree ran since
 * begin).  Each pointer is nullable, host or device; one launch.  TWIXT_EINVAL on a search created without
 * TWIXT_MCTS_SOLVE, before begin, or while a select awaits its backup. */
#define TWIXT_MCTS_PUCT 1u
#define TWIXT_MCTS_SOLVE 2u
#define TWIXT_MCTS_LEAF_SOLVED 2
#define TWIXT_MCTS_UNPROVEN (-128)
int twixt_mcts_create_ex(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                         double uct_c, uint32_t flags, twixt_mcts** out);
int twixt_mcts_solver_stats(twixt_mcts* m, uint8_t* out_proven, float* out_returns, int8_t* out_edge_values,
                            int32_t* out_simulations);

/* Several leaves per step with virtual loss (leaf parallelism, as in AlphaGo, Leela Zero and KataGo): not an
 * open_spiel behaviour but this search's own, which reduces to the searches above at leaves_per_step = 1.
 * twixt_mcts_create_parallel takes the flags of twixt_mcts_create_ex, K = leaves_per_step (1 <= K <= 4096 and
 * K <= max_simulations) and the virtual loss vl (finite, >= 0); K = 1 is exactly twixt_mcts_create_ex with the same
 * flags.  TWIXT_MCTS_SOLVE with K > 1 is TWIXT_EINVAL.  One STEP is K simulations of every tree:
 *  - every node has a virtual visit count V(s) and every edge V(a), both 0 between steps.  Descent j = 0 .. K-1 of
 *    a step is simulation k = (simulations since begin) + j, whose k keys the unvisited-edge draw and the rollout
 *    streams as above.  The descents of a tree run in order j; each sees the virtual counts of the earlier ones.
 *  - the leaf rule is unchanged: a descent stops at a terminal node or at a node with N(s) == 0 (real visits).
 *    UCT still expands a node on its second real visit, in select; PUCT in backup.  A descent may end at a leaf
 *    that an earlier descent of the step already took (a repeated leaf): it is an ordinary row with its own env,
 *    rollouts or caller value.
 *  - scores use n_eff = N(a) + V(a), N_eff(s) = N(s) + V(s) and w_eff = (V(a) > 0 ? W(a) - vl*V(a) : W(a)) in IEEE
 *    double without contraction: UCT's unvisited-edge draw counts the edges with n_eff == 0, otherwise edges score
 *    q + c*sqrt(ln N_eff(s) / n_eff) with q = w_eff / n_eff; PUCT scores (w_eff / n_eff or 0) +
 *    ((c*P)*sqrt(N_eff(s))) / (n_eff + 1), and an edge whose child is terminal still scores its outcome.  Ties as
 *    before.
 *  - after descent j picks its path, V += 1 on every edge and every node of the path and on the leaf.
 *  - backup takes rows j = 0 .. K-1 of each tree in order: row j removes its virtual visits and adds its value
 *    as above (W only ever receives real values).  A PUCT leaf is expanded by the LOWEST row whose leaf it is,
 *    with that row's priors; the priors of repeated leaves are ignored.
 *  - step 0: N(root) = 0, so every descent stops at the root; a PUCT root is expanded with the priors of row
 *    t*K + 0 of the first backup, which is where root Dirichlet noise goes.
 * Shapes: twixt_mcts_select writes descent j of tree t to env leaf_first + t*K + j (the range check covers count*K
 * envs) and out_leaf_status [count*K]; twixt_mcts_backup / _backup_priors take values [count*K, 2] and priors
 * [count*K, n*n] (host priors are checked on every row).  twixt_mcts_run(s) needs s to be a multiple of K and
 * queues s / K steps of three launches, the playout launch running K*R rollouts per tree.  max_simulations counts
 * simulations: each step, or select/backup pair, counts K.  root_stats and destroy are unchanged.  The arena
 * holds K paths, K leaf entries and K*R rollout slots per tree and a u16 V per node and per edge
 * (twixt_mcts.cuh); K = 1 allocates nothing more. */
int twixt_mcts_create_parallel(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                               double uct_c, uint32_t flags, int32_t leaves_per_step, double virtual_loss,
                               twixt_mcts** out);

/* Tree reuse across moves (as AlphaGo Zero, Leela Zero and KataGo do; open_spiel's MCTSBot has none, so this is
 * the search's own behaviour).  A caller that never calls twixt_mcts_advance gets exactly the searches above.
 * twixt_mcts_advance(m, actions, keep_nodes, out_status): actions [count] int32 on the host or the device,
 * 1 <= keep_nodes <= S = max_simulations + 1, out_status [count] int32 (nullable).  For tree t:
 *  - a legal action whose root edge has a child: that child becomes the new root.  The kept nodes are its
 *    subtree, renumbered by their rank in old slot order (the new root is slot 0, children stay above their
 *    parents), each with all its data: record, N(s), legal count and its edges' action, N, W, child (remapped),
 *    prior, tie key and outcome code.  The node count becomes the number of kept nodes.
 *  - the cap: only the first keep_nodes nodes of that order are kept (still a rooted tree).  An edge whose child
 *    the cap drops is unvisited again (N = 0, W = 0, no child; prior, tie key and outcome code stay); its parent's
 *    N(s) is unchanged, and a later simulation that takes it creates the child afresh.
 *  - a legal action without a child (the edge was never taken, or the root is not expanded): the tree is cleared
 *    to the root with the move applied, as twixt_mcts_begin would from that state.
 *  - action -1: the tree keeps its root and is only cut to keep_nodes (finished self-play games).
 *  - an illegal action, which includes anything but -1 at a terminal root: the tree is unchanged and gets status
 *    1, and the call fails with TWIXT_EILLEGAL "Not a legal action: %d" exactly as twixt_apply reports it (with a
 *    device out_status the call returns at once and the statuses are the report; begin such a tree again before
 *    it runs more simulations, since the host's node bound below assumes every tree was cut to keep_nodes).
 *  - statuses: TWIXT_MCTS_ROOT_KEPT (0) the new root has statistics (N(root) > 0), TWIXT_MCTS_ROOT_ILLEGAL (1),
 *    TWIXT_MCTS_ROOT_FRESH (2) the new root has none (N(root) = 0): the next simulation evaluates it.
 *  - solver searches: the new root's code is 4 - c from the chosen edge's code c != 0 (the child's value for its
 *    own player to move), else 0; a tree advanced into a proven child stays finished.
 *  - the stream id T and the simulation counter k, which key the unvisited-edge draw and the rollout streams,
 *    carry on across advances, so a tree never repeats a Philox counter.
 * It is TWIXT_EINVAL before begin and while a select is pending, and works with every kind and with K > 1.  One
 * launch; the first call allocates an int32 slot map of count x S entries (not part of the create-time arena).
 * Budget, without host synchronisation: the host bounds the node count (1 after begin, min(keep_nodes, bound)
 * after an advance, +K per step) and run(s) / select fail with TWIXT_EINVAL when bound + s > S; without an
 * advance this is the "more than max_simulations simulations since begin" check.  k*R + r must stay below 2^32.
 * Size the arena for reuse: max_simulations = the capacity, e.g. 2*sims with keep_nodes = sims + 1 runs sims new
 * simulations every move.
 * twixt_mcts_set_root_priors(m, priors [count, n*n] float32, host or device), PUCT only: replaces P(a) on every
 * root edge of each tree whose root is expanded; other trees are left alone (their first backup still takes the
 * priors of row t*K + 0).  This is how root Dirichlet noise reaches a kept root.  Host priors are checked as
 * twixt_mcts_backup_priors checks them.  TWIXT_EINVAL on a UCT search, before begin or while a select is pending.
 * One launch. */
#define TWIXT_MCTS_ROOT_KEPT 0
#define TWIXT_MCTS_ROOT_ILLEGAL 1
#define TWIXT_MCTS_ROOT_FRESH 2
int twixt_mcts_advance(twixt_mcts* m, const int32_t* actions, int32_t keep_nodes, int32_t* out_status);
int twixt_mcts_set_root_priors(twixt_mcts* m, const float* priors);

/* Gumbel AlphaZero search (Danihelka, Guez, Schrittwieser, Silver, "Policy improvement by planning with Gumbel",
 * ICLR 2022; mctx gumbel_muzero_policy with qtransform_completed_by_mix_value's defaults), in reproducible IEEE
 * double instead of float32.  The tree is the PUCT one: one node per simulation in creation order, edges the legal
 * actions ascending, a leaf at a terminal node or a node with N(s) == 0, expanded at its backup, and the backup adds
 * v[player to move at the parent] to W(a) along the path.  What differs:
 *  - every edge carries a float32 logit l(a): the backup's [count, n*n] array (the priors of twixt_mcts_backup_priors
 *    are read as logits), or 0 for every edge without one (twixt_mcts_run, twixt_mcts_backup, a NULL pointer).
 *    Entries of illegal actions are ignored; host logits must be finite on the legal actions of every non-terminal
 *    leaf (checked on the host against the leaf envs select wrote; TWIXT_EINVAL, trees unchanged).
 *  - every node keeps its raw value v(s): its evaluation for its own player to move (the caller's value, the
 *    rollout mean, or Returns() of a terminal leaf).
 *  - the completed Q at a node s: pi = softmax(l) raised to the smallest normal double, q(a) = W(a)/N(a) on visited
 *    edges, SN = sum N(a), v_mix = (v(s) + SN * sum_{N>0} (pi*q / sum_{N>0} pi)) / (SN + 1), q~ = q on visited
 *    edges and v_mix elsewhere, q^ = (q~ - min q~) / max(max q~ - min q~, 1e-8), sigma = ((c_visit + max N) *
 *    c_scale) * q^.
 *  - interior nodes take argmax of softmax(l + sigma)(a) - N(a) / (1 + SN), ties to the lower edge.
 *  - the root takes Sequential Halving: m = min(max_considered, L), i = SN (= N(root) - 1); the eligible edges have
 *    N(a) = table[m][i] with table = mctx's get_table_of_considered_visits(max_considered, max_simulations - 1);
 *    among them argmax of max(-1e9, (g(a) + (l(a) - max l)) + sigma(a)), ties to the lower edge.
 *  - g is the root's Gumbel noise per action cell, zeroed by begin (mctx's gumbel_scale = 0) and set by
 *    twixt_mcts_set_root_gumbel(m, gumbel [count, n*n] float32, host or device; host values must be finite).
 *  - every exp and every sum over a node's edges is fixed bit for bit (twixt_mcts.cuh: mcts_exp, mcts_lane_sums).
 * twixt_mcts_create_gumbel: max_considered >= 1 (above n(n-2) it acts as n(n-2)), c_visit (mctx maxvisit_init, 50)
 * and c_scale (mctx value_scale, 0.1) finite and >= 0, else TWIXT_EINVAL.  A Gumbel search has no solver and one
 * leaf per step, and twixt_mcts_advance and twixt_mcts_set_root_priors on it are TWIXT_EINVAL (Sequential Halving
 * assumes a fresh root).  begin, run, select, backup and backup_priors work as above with the same launch counts.
 * twixt_mcts_root_stats returns visits and value sums as for every kind, and out_best is the Gumbel action (one
 * more launch).
 * twixt_mcts_gumbel_stats: out_action [count] int32, the root score above among the edges with N(a) = max N (-1 for
 * a terminal or unexpanded root), and out_policy [count, n*n] float32, the improved policy softmax(l + sigma) at the
 * root's action cells, 0 elsewhere (all 0 for a terminal or unexpanded root; mctx's action_weights).  Each pointer
 * is nullable, host or device; one launch; TWIXT_EINVAL on another kind, before begin or while a select is pending.
 * Arena per tree: S*(rw*4 + 16 + 22*M) + 16 + 8*P + R*(rw*4 + 16) + 4*n*n bytes (a logit per edge, v per node,
 * the root noise), plus (min(max_considered, M) + 1) * (max_simulations - 1) int32 of table per search; TWIXT_ENOMEM
 * names it. */
int twixt_mcts_create_gumbel(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                             int32_t max_considered, double c_visit, double c_scale, twixt_mcts** out);
int twixt_mcts_set_root_gumbel(twixt_mcts* m, const float* gumbel);
int twixt_mcts_gumbel_stats(twixt_mcts* m, int32_t* out_action, float* out_policy);

/* Multi-GPU plumbing for hosts that are not Python (SURVEY 8e: envs shard by contiguous global id ranges,
 * no data-path collective, one reduction of the counters).  twixt_shard_range: rank's share [first,
 * first+count) of global_envs envs over `world` ranks (shares differ by at most one env); create the rank's
 * batch with `count` envs and call twixt_set_stream_base(b, first) so games do not depend on the GPU
 * count.  twixt_stats_accumulate: acc += part (sums; max for max_length) -- apply it to the ranks'
 * twixt_get_stats results, or to the output of an MPI/NCCL all-gather.  Neither needs a GPU. */
int twixt_shard_range(int64_t global_envs, int32_t world, int32_t rank, int64_t* out_first,
                      int64_t* out_count);
int twixt_stats_accumulate(twixt_stats* acc, const twixt_stats* part);

#ifdef __cplusplus
}
#endif
#endif /* TWIXT_B200_H_ */
