"""TEST INFRASTRUCTURE: executable specification of the batched MCTS search (include/twixt_b200.h, "Batched
MCTS"), written on the oracle (oracle/pyoracle.py) and nothing else.

It is open_spiel's MCTSBot with RandomRolloutEvaluator(R), solve = false and no Dirichlet noise, with the
changes that make it reproducible on the GPU: the one random draw per simulation (which unvisited edge to take)
comes from Philox counter (T lo, T hi, k, 1), the rollouts are the fused playout's Philox streams
(T << 32) | (k*R + r), the UCT score is evaluated in IEEE double as q = W/N, e = c*sqrt(log(N(s))/N), q + e,
and ties go to the lowest action.  Nodes are numbered in creation order (root 0), one new node per simulation
at most, as the device arena stores them.
"""
from __future__ import annotations

import math
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from oracle import pyoracle

M32 = 0xFFFFFFFF


class Node:
    __slots__ = ("state", "n", "actions", "edge_n", "edge_w", "children", "parent", "action")

    def __init__(self, state, parent: int, action: int):
        self.state = state
        self.n = 0
        self.actions: Optional[List[int]] = None  # None until expanded
        self.edge_n: List[int] = []
        self.edge_w: List[float] = []
        self.children: List[int] = []
        self.parent = parent
        self.action = action


def uct_score(w: float, n: int, parent_visits: int, c: float) -> float:
    q = w / n
    e = c * math.sqrt(math.log(parent_visits) / n)
    return q + e


def draw(seed: int, tree_stream: int, k: int, unvisited: int) -> int:
    word = pyoracle.philox([tree_stream & M32, tree_stream >> 32, k, 1], [seed & M32, (seed >> 32) & M32])[0]
    return (word * unvisited) >> 32


def rollout_stream(tree_stream: int, k: int, R: int, r: int) -> int:
    return (tree_stream << 32) | (k * R + r)


class Search:
    """One tree.  `root` is an OracleState (copied)."""

    def __init__(self, root, seed: int, tree_stream: int, n_rollouts: int = 1, uct_c: float = 2.0):
        if tree_stream >= 1 << 32:
            raise ValueError("tree stream id must be below 2^32")
        self.seed = seed
        self.T = tree_stream
        self.R = n_rollouts
        self.c = float(uct_c)
        self.nodes: List[Node] = [Node(root.clone(), -1, -1)]
        self.k = 0
        self._pending: Optional[Tuple[List[Tuple[int, int]], int]] = None

    # -- one simulation in two halves (the stepwise form) ------------------------------------------------------
    def select(self) -> Tuple[int, bool]:
        """Descends; returns (leaf node index, leaf is terminal).  The path is kept for backup()."""
        assert self._pending is None
        path: List[Tuple[int, int]] = []  # (node, edge)
        s = 0
        while True:
            node = self.nodes[s]
            if node.state.is_terminal() or node.n == 0:
                break
            if node.actions is None:
                node.actions = node.state.legal_actions()
                L = len(node.actions)
                node.edge_n, node.edge_w, node.children = [0] * L, [0.0] * L, [-1] * L
            unvisited = [i for i, v in enumerate(node.edge_n) if v == 0]
            if unvisited:
                e = unvisited[draw(self.seed, self.T, self.k, len(unvisited))]
            else:
                best, e = None, -1
                for i in range(len(node.actions)):
                    sc = uct_score(node.edge_w[i], node.edge_n[i], node.n, self.c)
                    if best is None or sc > best:
                        best, e = sc, i
            path.append((s, e))
            if node.children[e] < 0:
                child = node.state.clone()
                child.apply_action(node.actions[e])
                self.nodes.append(Node(child, s, node.actions[e]))
                node.children[e] = len(self.nodes) - 1
            s = node.children[e]
        self._pending = (path, s)
        return s, self.nodes[s].state.is_terminal()

    def backup(self, value: Optional[Sequence[float]] = None) -> None:
        """value: the leaf's [2] values (float32 in the stepwise form), ignored for a terminal leaf."""
        path, leaf = self._pending
        st = self.nodes[leaf].state
        if st.is_terminal():
            v = [float(x) for x in st.returns()]
        else:
            v = [float(value[0]), float(value[1])]
        for s, e in path:
            node = self.nodes[s]
            p = node.state.current_player()
            node.n += 1
            node.edge_n[e] += 1
            node.edge_w[e] += v[p]
        self.nodes[leaf].n += 1
        self._pending = None
        self.k += 1

    def rollout_value(self, leaf: int) -> List[float]:
        """RandomRolloutEvaluator: the mean of R fused playouts, summed in double, r ascending."""
        sums = [0.0, 0.0]
        for r in range(self.R):
            st = self.nodes[leaf].state.clone()
            st.playout_philox(self.seed, rollout_stream(self.T, self.k, self.R, r))
            ret = st.returns()
            sums[0] += ret[0]
            sums[1] += ret[1]
        return [sums[0] / self.R, sums[1] / self.R]

    def simulate(self, value_fn: Optional[Callable] = None) -> None:
        leaf, terminal = self.select()
        if terminal:
            self.backup(None)
        elif value_fn is None:
            self.backup(self.rollout_value(leaf))
        else:
            self.backup(value_fn(self.nodes[leaf].state.export_record()))

    def run(self, num_simulations: int, value_fn: Optional[Callable] = None) -> "Search":
        for _ in range(num_simulations):
            self.simulate(value_fn)
        return self

    # -- results ------------------------------------------------------------------------------------------------
    def root_stats(self, n: int) -> Tuple[np.ndarray, np.ndarray, int]:
        """(visits [n*n] int32, value_sums [n*n] float64, best action or -1) as twixt_mcts_root_stats."""
        root = self.nodes[0]
        visits = np.zeros(n * n, dtype=np.int32)
        sums = np.zeros(n * n, dtype=np.float64)
        best = -1
        if root.actions:
            bi = 0
            for i, a in enumerate(root.actions):
                visits[a] = root.edge_n[i]
                sums[a] = root.edge_w[i]
                if (root.edge_n[i], root.edge_w[i]) > (root.edge_n[bi], root.edge_w[bi]):
                    bi = i
            best = root.actions[bi]
        return visits, sums, best


def stand_in_value(record: np.ndarray) -> np.ndarray:
    """A deterministic value of a leaf record for the stepwise tests: float32 in [-1, 1] per player."""
    h = int(np.bitwise_xor.reduce(record.astype(np.uint64) * np.uint64(2654435761) + np.arange(record.size,
                                                                                                   dtype=np.uint64)))
    a = ((h & 0xFFFF) % 2001 - 1000) / 1000.0
    b = (((h >> 16) & 0xFFFF) % 2001 - 1000) / 1000.0
    return np.asarray([a, b], dtype=np.float32)


def root_positions(game, n: int, seed: int, count: int) -> List[object]:
    """Roots of every kind the tests want, cycled: ply 0, ply 1 (swap offer), mid-game, one move before the
    end, terminal, and a draw-bound position (late in a game with few legal cells left)."""
    import random
    rng = random.Random(seed)
    out = []
    for i in range(count):
        kind = i % 6
        st = game.new_initial_state()
        if kind == 1:
            st.apply_action(rng.choice(st.legal_actions()))
        elif kind == 2:
            for _ in range(rng.randrange(3, max(4, n * n // 4))):
                if st.is_terminal():
                    break
                st.apply_action(rng.choice(st.legal_actions()))
        elif kind in (3, 4, 5):
            full = st.clone()
            acts = full.playout_philox(seed, 1000 + i)
            keep = {3: len(acts) - 1, 4: len(acts), 5: max(0, len(acts) - 3)}[kind]
            for a in acts[:keep]:
                st.apply_action(a)
        out.append(st)
    return out
