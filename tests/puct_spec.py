"""TEST INFRASTRUCTURE: executable specification of the PUCT search (include/twixt_b200.h, "PUCT search with
policy priors"), written on the oracle (oracle/pyoracle.py) and nothing else.

It restates open_spiel's python/algorithms/mcts.py -- SearchNode.puct_value, SearchNode.sort_key,
_apply_tree_policy and mcts_search -- for MCTSBot(child_selection_fn=puct_value, solve=False), with the
substitutions that make it reproducible on the GPU:
  * a non-terminal leaf is expanded at its backup, with the priors that came with its value (open_spiel expands
    it on its second visit from evaluator.prior, which AlphaZeroEvaluator answers from the same network call);
    without priors P(a) = float32(1 / L), RandomRolloutEvaluator.prior;
  * priors are stored as float32;
  * the shuffle of the children at expansion is the order of their tie keys: word 0 of Philox4x32-10(key = seed,
    counter = (T, node slot, edge index, 2)), then the edge index;
  * the built-in evaluator's rollouts are the fused playout's Philox streams (T << 32) | (k*R + r).
Nodes are numbered in creation order (root 0), one new node per simulation at most, as the device arena stores
them; edges are the legal actions in ascending order.
"""
from __future__ import annotations

import math
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from oracle import pyoracle

M32 = 0xFFFFFFFF


def tie_key(seed: int, tree_stream: int, slot: int, edge: int) -> int:
    return pyoracle.philox([tree_stream & M32, slot, edge, 2], [seed & M32, (seed >> 32) & M32])[0]


def f32(x: float) -> float:
    return float(np.float32(x))


class SearchNode:
    """open_spiel's SearchNode.  `edge` is the child's index in its parent's ascending legal list, `key` its tie
    key, `slot` its creation-order slot (None until a simulation first reaches it), `state` its state then."""
    __slots__ = ("action", "player", "prior", "explore_count", "total_reward", "outcome", "children", "edge", "key",
                 "slot", "state", "parent_slot")

    def __init__(self, action, player, prior, edge=-1, key=0):
        self.action = action
        self.player = player
        self.prior = prior
        self.explore_count = 0
        self.total_reward = 0.0
        self.outcome = None
        self.children: List["SearchNode"] = []  # in shuffled (tie key) order
        self.edge = edge
        self.key = key
        self.slot = None
        self.state = None
        self.parent_slot = -1

    def puct_value(self, parent_explore_count, uct_c):
        if self.outcome is not None:
            return self.outcome[self.player]
        return ((self.explore_count and self.total_reward / self.explore_count) +
                uct_c * self.prior * math.sqrt(parent_explore_count) / (self.explore_count + 1))

    def sort_key(self):
        return (0 if self.outcome is None else self.outcome[self.player], self.explore_count, self.total_reward)

    def edges(self) -> List["SearchNode"]:
        """The children in ascending action order (the device's edge order)."""
        return sorted(self.children, key=lambda c: c.edge)


class Search:
    """One tree.  `root` is an OracleState (copied)."""

    def __init__(self, root, seed: int, tree_stream: int, n_rollouts: int = 1, uct_c: float = 2.0):
        if tree_stream >= 1 << 32:
            raise ValueError("tree stream id must be below 2^32")
        self.seed = seed
        self.T = tree_stream
        self.R = n_rollouts
        self.c = float(uct_c)
        r = SearchNode(None, max(root.current_player(), 0), 1.0)  # a terminal root's player is never read
        r.slot, r.state = 0, root.clone()
        self.nodes: List[SearchNode] = [r]  # by slot
        self.k = 0
        self._pending = None

    # -- _apply_tree_policy: descend to a terminal node or one that has not been explored ----------------------
    def select(self) -> Tuple[int, bool]:
        assert self._pending is None
        current = self.nodes[0]
        visit_path = [current]
        while not current.state.is_terminal() and current.explore_count > 0:
            chosen = max(current.children, key=lambda c: c.puct_value(current.explore_count, self.c))
            if chosen.slot is None:
                chosen.state = current.state.clone()
                chosen.state.apply_action(chosen.action)
                chosen.slot = len(self.nodes)
                chosen.parent_slot = current.slot
                self.nodes.append(chosen)
            current = chosen
            visit_path.append(current)
        self._pending = visit_path
        return current.slot, current.state.is_terminal()

    # -- mcts_search's backup, then the expansion of a non-terminal leaf with its priors -------------------------
    def backup(self, value: Optional[Sequence[float]] = None, priors: Optional[Sequence[float]] = None) -> None:
        """value: the leaf's [2] values (float32 in the stepwise form); priors: [n*n] or None (uniform).  Both
        are ignored for a terminal leaf."""
        visit_path = self._pending
        leaf = visit_path[-1]
        st = leaf.state
        if st.is_terminal():
            returns = [float(x) for x in st.returns()]
            leaf.outcome = returns
        else:
            returns = [float(value[0]), float(value[1])]
        for node in visit_path:
            node.total_reward += returns[node.player]  # the root's sum is not observable
            node.explore_count += 1
        if not st.is_terminal():
            legal = st.legal_actions()
            player = st.current_player()
            kids = []
            for i, a in enumerate(legal):
                p = f32(1.0 / len(legal)) if priors is None else f32(priors[a])
                kids.append(SearchNode(a, player, p, i, tie_key(self.seed, self.T, leaf.slot, i)))
            leaf.children = sorted(kids, key=lambda c: (c.key, c.edge))  # "shuffle"
        self._pending = None
        self.k += 1

    def rollout_value(self, leaf: int) -> List[float]:
        """RandomRolloutEvaluator: the mean of R fused playouts, summed in double, r ascending."""
        sums = [0.0, 0.0]
        for r in range(self.R):
            st = self.nodes[leaf].state.clone()
            st.playout_philox(self.seed, (self.T << 32) | (self.k * self.R + r))
            ret = st.returns()
            sums[0] += ret[0]
            sums[1] += ret[1]
        return [sums[0] / self.R, sums[1] / self.R]

    def simulate(self, value_fn: Optional[Callable] = None, prior_fn: Optional[Callable] = None) -> None:
        leaf, terminal = self.select()
        if terminal:
            self.backup(None)
            return
        rec = self.nodes[leaf].state.export_record()
        value = self.rollout_value(leaf) if value_fn is None else value_fn(rec)
        self.backup(value, None if prior_fn is None else prior_fn(rec))

    def run(self, num_simulations: int, value_fn: Optional[Callable] = None,
            prior_fn: Optional[Callable] = None) -> "Search":
        for _ in range(num_simulations):
            self.simulate(value_fn, prior_fn)
        return self

    # -- results ------------------------------------------------------------------------------------------------
    def best_child(self) -> Optional[SearchNode]:
        root = self.nodes[0]
        if not any(c.explore_count > 0 for c in root.children):
            return None
        return max(root.children, key=SearchNode.sort_key)

    def root_stats(self, n: int) -> Tuple[np.ndarray, np.ndarray, int]:
        """(visits [n*n] int32, value_sums [n*n] float64, best action or -1) as twixt_mcts_root_stats."""
        visits = np.zeros(n * n, dtype=np.int32)
        sums = np.zeros(n * n, dtype=np.float64)
        for c in self.nodes[0].children:
            visits[c.action] = c.explore_count
            sums[c.action] = c.total_reward
        b = self.best_child()
        return visits, sums, -1 if b is None else b.action

    def dump(self):
        """Per slot: (parent slot, action, N(s), edge count or -1, [N(a)], [W(a)], [P(a)]) in edge order."""
        out = []
        for node in self.nodes:
            e = node.edges()
            L = len(e) if node.children else -1
            out.append((node.parent_slot, -1 if node.action is None else node.action, node.explore_count, L,
                        [c.explore_count for c in e], [c.total_reward for c in e], [c.prior for c in e]))
        return out


def stand_in_priors(record: np.ndarray, n: int) -> np.ndarray:
    """A deterministic float32 distribution [n*n] computed from a leaf record for the stepwise tests: a hashed
    weight in 1..64 on every cell without a peg and on the first move's cell (the swap offer), 0 elsewhere,
    normalised.  It is positive on every legal action and also on a few illegal ones (the border cells the
    player to move may not use), which the search must ignore."""
    rec = record.astype(np.uint64)
    h = int(np.bitwise_xor.reduce(rec * np.uint64(0x9E3779B1) + np.arange(rec.size, dtype=np.uint64) * np.uint64(7)))
    cells = np.arange(n * n, dtype=np.uint64)
    w = ((cells * np.uint64(0x85EBCA6B) + np.uint64(h & 0xFFFFFFFF)) >> np.uint64(7)) % np.uint64(64) + np.uint64(1)
    w = w.astype(np.float64)
    x, y = np.divmod(np.arange(n * n), n)
    red, blue = record[4 + x].astype(np.int64), record[4 + n + x].astype(np.int64)
    occupied = (((red | blue) >> y) & 1).astype(bool)
    first = int(record[2])
    keep = ~occupied
    if record[0] == 1 and first != 0xFFFFFFFF:
        keep[first] = True
    w[~keep] = 0.0
    return (w / w.sum()).astype(np.float32)
