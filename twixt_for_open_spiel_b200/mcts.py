"""Batched MCTS on the device (twixt_mcts_* in include/twixt_b200.h, kernels in csrc/twixt_mcts.cu).

`BatchedMCTS` runs thousands of independent UCT searches at once, one tree per root env of a `TwixTBatch`:
open_spiel's MCTSBot with RandomRolloutEvaluator(n_rollouts), solve = false and no Dirichlet noise, made
deterministic (the header describes every draw).  The whole tree lives in HBM; a simulation is three kernel
launches (select, fused playouts, backup) for all trees together.

Two ways to evaluate leaves:
  * built in:  `run(k)` -- R random rollouts per leaf with the fused playout kernel;
  * stepwise:  `select(leaf_first)` copies every tree's leaf into batch envs [leaf_first, leaf_first + count),
    the caller evaluates them (e.g. `observation_and_mask` + a value network) and hands the values to
    `backup(values)`.

`selection="puct"` makes every tree open_spiel's AlphaZero search instead (MCTSBot with
child_selection_fn = puct_value): `backup(values, priors)` hands the policy head's priors [count, n*n] with
the values, and the leaf is expanded with them.  `add_dirichlet_noise` mixes open_spiel's root noise into the
priors of the first backup after `begin` (simulation 0's leaf is always the root; with leaves_per_step = K, row
t*K + 0 of that backup).

`solve=True` adds open_spiel's MCTS-Solver to either kind (MCTSBot(..., solve=True), open_spiel's default):
a terminal leaf proves nodes up its path, a proven child is scored by its outcome, and a tree whose root is
proven is finished: later simulations do nothing for it (`select` reports LEAF_SOLVED and leaves its env
alone).  `solver_stats()` returns the proven root and move values.

`leaves_per_step=K` (K > 1) descends K times per tree in one step, with virtual loss steering the later descents
of a step away from the earlier ones (leaf parallelism, as in AlphaGo, Leela Zero and KataGo; not an open_spiel
behaviour, and exactly the search above at K = 1).  All K leaves of every tree are evaluated together: `run`
plays K*R rollouts per tree in one playout launch, and the stepwise form hands the caller K rows per tree, so a
search needs max_simulations / K steps instead of max_simulations.  Row t*K + j is descent j of tree t.

`advance(actions, keep_nodes)` reuses the trees across moves (as AlphaGo Zero, Leela Zero and KataGo do; not an
open_spiel behaviour): the child of each root along the move played becomes the new root with its subtree and all
its statistics, up to keep_nodes nodes, so the next search starts from the visits the last one already spent there.
Size the search for it: max_simulations is the node capacity, e.g. 2*sims with keep_nodes = sims + 1 runs sims new
simulations every move.  `set_root_priors` puts fresh priors (root Dirichlet noise) on the kept roots.

`MCTSBot` is the open_spiel-shaped bot over one tree for adapter `TwixTState`s.

Arrays may be numpy (synchronous) or torch CUDA tensors (asynchronous on the batch's stream), as for
`TwixTBatch`.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib
from .batch import TwixTBatch, _dt, _is_torch, _ptr

LEAF_NEEDS_VALUE, LEAF_TERMINAL, LEAF_SOLVED = 0, 1, 2
ROOT_KEPT, ROOT_ILLEGAL, ROOT_FRESH = 0, 1, 2  # advance(): statistics kept, illegal action, new root unvisited
UNPROVEN = -128  # solver_stats' edge value of a root move that is not proven
_PUCT, _SOLVE = 1, 2  # TWIXT_MCTS_PUCT, TWIXT_MCTS_SOLVE


class BatchedMCTS:
    def __init__(self, batch: TwixTBatch, num_trees: int, max_simulations: int, n_rollouts: int = 1,
                 uct_c: float = 2.0, selection: str = "uct", solve: bool = False, leaves_per_step: int = 1,
                 virtual_loss: float = 1.0):
        if selection not in ("uct", "puct"):
            raise ValueError("selection must be 'uct' or 'puct', got %r" % (selection,))
        self._lib = _lib.load()
        self.batch = batch  # the search runs on the batch's envs and stream: keep it alive
        self._h = C.c_void_p()
        flags = (_PUCT if selection == "puct" else 0) | (_SOLVE if solve else 0)
        if int(leaves_per_step) == 1:
            self._check(self._lib.twixt_mcts_create_ex(batch._h, int(num_trees), int(max_simulations),
                                                       int(n_rollouts), float(uct_c), flags, C.byref(self._h)))
        else:
            self._check(self._lib.twixt_mcts_create_parallel(
                batch._h, int(num_trees), int(max_simulations), int(n_rollouts), float(uct_c), flags,
                int(leaves_per_step), float(virtual_loss), C.byref(self._h)))
        self.leaves_per_step = int(leaves_per_step)
        self.virtual_loss = float(virtual_loss)
        self.selection = selection
        self.solve = bool(solve)
        self.num_trees = int(num_trees)
        self.max_simulations = int(max_simulations)
        self.n_rollouts = int(n_rollouts)
        self.uct_c = float(uct_c)
        self.count = 0
        self._cells = batch.board_size * batch.board_size

    def _check(self, rc: int):
        if rc != 0:
            self.batch._raise(rc)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            # a search must be destroyed before its batch; when the garbage collector finalises a cycle that holds
            # both (a failed test's frame, interpreter exit) the batch may go first, and the search's device memory
            # is then left to the process's exit rather than freed through the batch's released stream
            if self.batch._h.value:
                self._lib.twixt_mcts_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def begin(self, first: int = 0, count: Optional[int] = None):
        """Copies envs [first, first + count) as the roots of trees [0, count) and clears the trees."""
        if count is None:
            count = self.num_trees
        self._check(self._lib.twixt_mcts_begin(self._h, int(first), int(count)))
        self.count = int(count)

    def run(self, num_simulations: int):
        """num_simulations simulations of every tree with the built-in rollout evaluator (asynchronous); a
        multiple of leaves_per_step."""
        self._check(self._lib.twixt_mcts_run(self._h, int(num_simulations)))

    def select(self, leaf_first: int, out_status=None):
        """Stepwise form, first half: leaf of descent j of tree t -> batch env leaf_first + t*K + j (K =
        leaves_per_step; t with K = 1).  Returns the statuses [count*K] int32 (LEAF_NEEDS_VALUE, or LEAF_TERMINAL:
        its value is Returns() and backup ignores the caller's, or with solve=True LEAF_SOLVED: the tree is
        finished, its env was not written and backup ignores its row)."""
        rows = self.count * self.leaves_per_step
        if out_status is None:
            out_status = np.zeros(rows, dtype=np.int32)
        self._check(self._lib.twixt_mcts_select(self._h, int(leaf_first),
                                                _ptr(out_status, _dt(np.int32, "int32"), rows)))
        return out_status

    def backup(self, values, priors=None):
        """Stepwise form, second half: values [count*K, 2] float32 of the leaves select() wrote.  A PUCT search
        also takes priors [count*K, n*n] float32 (None: uniform over the legal actions); entries of illegal
        actions, rows of terminal leaves and (K > 1) the rows of repeated leaves after the first are ignored."""
        rows = self.count * self.leaves_per_step
        if not _is_torch(values):
            values = np.ascontiguousarray(values, dtype=np.float32)
        if priors is not None and not _is_torch(priors):
            priors = np.ascontiguousarray(priors, dtype=np.float32)
        self._check(self._lib.twixt_mcts_backup_priors(
            self._h, _ptr(values, _dt(np.float32, "float32"), 2 * rows),
            _ptr(priors, _dt(np.float32, "float32"), rows * self._cells)))

    def root_stats(self, out_visits=None, out_value_sums=None, out_best=None):
        """(visits [count, n*n] int32, value_sums [count, n*n] float64, best [count] int32) of the root edges;
        best is -1 where the root is terminal or not yet expanded (PUCT: while no root edge has a visit)."""
        if out_visits is None:
            out_visits = np.zeros((self.count, self._cells), dtype=np.int32)
        if out_value_sums is None:
            out_value_sums = np.zeros((self.count, self._cells), dtype=np.float64)
        if out_best is None:
            out_best = np.zeros(self.count, dtype=np.int32)
        self._check(self._lib.twixt_mcts_root_stats(
            self._h, _ptr(out_visits, _dt(np.int32, "int32"), self.count * self._cells),
            _ptr(out_value_sums, _dt(np.float64, "float64"), self.count * self._cells),
            _ptr(out_best, _dt(np.int32, "int32"), self.count)))
        return out_visits, out_value_sums, out_best

    def best(self) -> np.ndarray:
        return self.root_stats()[2]

    def solver_stats(self, out_proven=None, out_returns=None, out_edge_values=None, out_simulations=None):
        """solve=True only: (proven [count] uint8, returns [count, 2] float32, edge_values [count, n*n] int8,
        simulations [count] int32).  proven is 1 once the root is proven; returns is open_spiel's root.outcome
        ((0, 0) while unproven); edge_values is -1, 0 or +1 for a proven root move from the view of the player to
        move at the root, UNPROVEN elsewhere; simulations is N(root), the simulations the tree ran since begin
        (a finished tree stops counting)."""
        if out_proven is None:
            out_proven = np.zeros(self.count, dtype=np.uint8)
        if out_returns is None:
            out_returns = np.zeros((self.count, 2), dtype=np.float32)
        if out_edge_values is None:
            out_edge_values = np.zeros((self.count, self._cells), dtype=np.int8)
        if out_simulations is None:
            out_simulations = np.zeros(self.count, dtype=np.int32)
        self._check(self._lib.twixt_mcts_solver_stats(
            self._h, _ptr(out_proven, _dt(np.uint8, "uint8"), self.count),
            _ptr(out_returns, _dt(np.float32, "float32"), 2 * self.count),
            _ptr(out_edge_values, _dt(np.int8, "int8"), self.count * self._cells),
            _ptr(out_simulations, _dt(np.int32, "int32"), self.count)))
        return out_proven, out_returns, out_edge_values, out_simulations

    def advance(self, actions, keep_nodes: Optional[int] = None, out_status=None):
        """Tree reuse: actions [count] int32 (the move played in each tree's root, -1 to keep the root).  The child
        along the move becomes the new root with its subtree and all its statistics, at most keep_nodes nodes of it
        (None: max_simulations + 1, all of them); a move whose edge has no child clears the tree to the new
        position.  Returns the statuses [count] int32: ROOT_KEPT (the new root has visits), ROOT_FRESH (it has
        none: the next simulation evaluates it) or ROOT_ILLEGAL.  An illegal move leaves its tree unchanged and
        raises, as `TwixTBatch.apply` does, unless out_status is a torch CUDA tensor (asynchronous: the statuses
        are the report).  The simulation counter carries on, so the draws never repeat."""
        if keep_nodes is None:
            keep_nodes = self.max_simulations + 1
        if not _is_torch(actions):
            actions = np.ascontiguousarray(np.reshape(actions, -1), dtype=np.int32)
        if out_status is None:
            out_status = np.zeros(self.count, dtype=np.int32)
        self._check(self._lib.twixt_mcts_advance(self._h, _ptr(actions, _dt(np.int32, "int32"), self.count),
                                                 int(keep_nodes), _ptr(out_status, _dt(np.int32, "int32"),
                                                                       self.count)))
        return out_status

    def set_root_priors(self, priors):
        """PUCT only: replaces P(a) of every root edge of each tree whose root is expanded with priors [count, n*n]
        float32 (e.g. root Dirichlet noise after `advance`).  Trees whose root is not expanded are left alone: their
        first backup takes the priors of row t*K + 0 as after `begin`."""
        if not _is_torch(priors):
            priors = np.ascontiguousarray(priors, dtype=np.float32)
        self._check(self._lib.twixt_mcts_set_root_priors(
            self._h, _ptr(priors, _dt(np.float32, "float32"), self.count * self._cells)))


def add_dirichlet_noise(priors, legal_mask, epsilon: float, alpha: float):
    """open_spiel's root noise: (1 - epsilon) * p + epsilon * Dir(alpha) over each row's legal actions.

    It goes into the priors of the first backup after `begin`, whose rows are the roots.  With leaves_per_step =
    K > 1 every descent of that first step stops at the root and the root takes the priors of row t*K + 0, so
    noise belongs in the rows t*K + 0 (the other rows' priors for the root are ignored).

    priors [B, A] float32 and legal_mask [B, A] (bool or 0/1) are torch tensors on the CPU or a GPU; returns a
    new float32 tensor on the same device.  Gamma(alpha) is drawn for every entry with torch's generator (so the
    result is reproducible under torch.manual_seed), in float64, zeroed where illegal and normalised per row;
    the mix is done in float32 (open_spiel mixes in double).  Entries of illegal actions are returned
    unchanged.  A row whose legal draws all underflow to 0 gets uniform noise over its legal actions."""
    import torch
    legal = legal_mask.to(device=priors.device, dtype=torch.bool)
    conc = torch.full(priors.shape, float(alpha), dtype=torch.float64, device=priors.device)
    g = torch.where(legal, torch.distributions.Gamma(conc, torch.ones_like(conc)).sample(),
                    torch.zeros_like(conc))
    total = g.sum(dim=1, keepdim=True)
    uniform = legal.to(torch.float64) / legal.sum(dim=1, keepdim=True).clamp_min(1)
    noise = torch.where(total > 0, g / torch.where(total > 0, total, torch.ones_like(total)), uniform)
    mixed = (1.0 - float(epsilon)) * priors.float() + float(epsilon) * noise.float()
    return torch.where(legal, mixed, priors.float())


class MCTSBot:
    """open_spiel's MCTSBot with RandomRolloutEvaluator(n_rollouts), for adapter states: what
    `mcts_example --player1=mcts --rollout_count=4` plays.  Each step copies the state's record into a private
    one-tree batch and runs max_simulations simulations on the device.

    solve defaults to False here, so existing callers keep the search they had; open_spiel's MCTSBot and
    mcts_example default to solve=True, which is `MCTSBot(..., solve=True)`: a proven win is played at once and
    the search of a step ends when its root is proven.

    leaves_per_step=K > 1 searches the one tree K leaves at a time with virtual loss (BatchedMCTS above), in
    max_simulations / K steps per move; max_simulations must then be a multiple of K and at least 2*K (step 0
    only evaluates the root).  The default K = 1 is the bot above.

    reuse_tree=True keeps the tree between steps (BatchedMCTS.advance): the search holds 2*max_simulations nodes,
    and `step(state)` advances through the actions by which state.history() extends the history it last searched
    (its own move, then the opponent's), keeping max_simulations + 1 nodes, then runs max_simulations new
    simulations.  A history that does not extend the last one begins a fresh tree."""

    def __init__(self, game, uct_c: float = 2.0, max_simulations: int = 1000, n_rollouts: int = 4, seed: int = 0,
                 device: int = 0, solve: bool = False, leaves_per_step: int = 1, virtual_loss: float = 1.0,
                 reuse_tree: bool = False):
        if max_simulations < 2:
            raise ValueError("MCTSBot needs max_simulations >= 2: the first simulation only evaluates the root")
        if leaves_per_step > 1 and (max_simulations % leaves_per_step or max_simulations < 2 * leaves_per_step):
            raise ValueError("MCTSBot with leaves_per_step = %d needs max_simulations to be a multiple of it and at "
                             "least twice it, got %d" % (leaves_per_step, max_simulations))
        self._game = game
        self._batch = TwixTBatch(game.board_size(), 1, device, seed)
        self._batch.set_validation(False)  # records come from the adapter's own exports
        capacity = (2 if reuse_tree else 1) * int(max_simulations)
        self._mcts = BatchedMCTS(self._batch, 1, capacity, n_rollouts, uct_c, solve=solve,
                                 leaves_per_step=leaves_per_step, virtual_loss=virtual_loss)
        self.max_simulations = int(max_simulations)
        self.reuse_tree = bool(reuse_tree)
        self._searched = None  # the history of the state the tree's root holds (reuse_tree)

    def step(self, state) -> int:
        if state.is_terminal():
            raise ValueError("MCTSBot.step on a terminal state")
        history = list(state.history())
        last = self._searched
        if self.reuse_tree and last is not None and history[:len(last)] == last:
            for a in history[len(last):] or [-1]:
                self._mcts.advance([a], self.max_simulations + 1)
        else:
            self._batch.import_state(state.export_record(), 0)
            self._mcts.begin(0, 1)
        self._searched = history
        self._mcts.run(self.max_simulations)
        return int(self._mcts.best()[0])

    def close(self):
        self._mcts.close()
        self._batch.close()
