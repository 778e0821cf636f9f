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

LEAF_NEEDS_VALUE, LEAF_TERMINAL = 0, 1


class BatchedMCTS:
    def __init__(self, batch: TwixTBatch, num_trees: int, max_simulations: int, n_rollouts: int = 1,
                 uct_c: float = 2.0):
        self._lib = _lib.load()
        self.batch = batch  # the search runs on the batch's envs and stream: keep it alive
        self._h = C.c_void_p()
        self._check(self._lib.twixt_mcts_create(batch._h, int(num_trees), int(max_simulations), int(n_rollouts),
                                                float(uct_c), C.byref(self._h)))
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
        """num_simulations simulations of every tree with the built-in rollout evaluator (asynchronous)."""
        self._check(self._lib.twixt_mcts_run(self._h, int(num_simulations)))

    def select(self, leaf_first: int, out_status=None):
        """Stepwise form, first half: leaf of tree t -> batch env leaf_first + t.  Returns the statuses
        [count] int32 (LEAF_NEEDS_VALUE, or LEAF_TERMINAL: its value is Returns() and backup ignores the
        caller's)."""
        if out_status is None:
            out_status = np.zeros(self.count, dtype=np.int32)
        self._check(self._lib.twixt_mcts_select(self._h, int(leaf_first),
                                                _ptr(out_status, _dt(np.int32, "int32"), self.count)))
        return out_status

    def backup(self, values):
        """Stepwise form, second half: values [count, 2] float32 of the leaves select() wrote."""
        if not _is_torch(values):
            values = np.ascontiguousarray(values, dtype=np.float32)
        self._check(self._lib.twixt_mcts_backup(self._h, _ptr(values, _dt(np.float32, "float32"), 2 * self.count)))

    def root_stats(self, out_visits=None, out_value_sums=None, out_best=None):
        """(visits [count, n*n] int32, value_sums [count, n*n] float64, best [count] int32) of the root edges;
        best is -1 where the root is terminal or not yet expanded."""
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


class MCTSBot:
    """open_spiel's MCTSBot with RandomRolloutEvaluator(n_rollouts), solve = false, for adapter states:
    what `mcts_example --player1=mcts --rollout_count=4` plays, without the solver.  Each step copies the
    state's record into a private one-tree batch and runs max_simulations simulations on the device."""

    def __init__(self, game, uct_c: float = 2.0, max_simulations: int = 1000, n_rollouts: int = 4, seed: int = 0,
                 device: int = 0):
        if max_simulations < 2:
            raise ValueError("MCTSBot needs max_simulations >= 2: the first simulation only evaluates the root")
        self._game = game
        self._batch = TwixTBatch(game.board_size(), 1, device, seed)
        self._batch.set_validation(False)  # records come from the adapter's own exports
        self._mcts = BatchedMCTS(self._batch, 1, max_simulations, n_rollouts, uct_c)
        self.max_simulations = int(max_simulations)

    def step(self, state) -> int:
        if state.is_terminal():
            raise ValueError("MCTSBot.step on a terminal state")
        self._batch.import_state(state.export_record(), 0)
        self._mcts.begin(0, 1)
        self._mcts.run(self.max_simulations)
        return int(self._mcts.best()[0])

    def close(self):
        self._mcts.close()
        self._batch.close()
