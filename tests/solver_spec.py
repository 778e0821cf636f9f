"""TEST INFRASTRUCTURE: executable specification of the MCTS-Solver searches (include/twixt_b200.h, "MCTS-Solver",
TWIXT_MCTS_SOLVE), written on the oracle and on the two specifications it extends, tests/mcts_spec.py (UCT) and
tests/puct_spec.py (PUCT), and nothing else.

It restates what open_spiel's python/algorithms/mcts.py adds with solve=True: in mcts_search, a terminal leaf
takes outcome = Returns(), and the backup walks the visit path up from it; a node whose children include one whose
outcome is max_utility for the node's player to move, or whose children all have outcomes, takes the best child's
outcome; the walk stops at the first node that takes none.  Selection scores a child with an outcome by
outcome[player] (uct_value, puct_value), and the best child is sort_key's (outcome or 0, N, W).  Once the root has
an outcome the tree's search ends: later simulations take no path (status LEAF_SOLVED), evaluate nothing and
change nothing but the simulation counter k.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np

import mcts_spec
import puct_spec

LEAF_NEEDS_VALUE, LEAF_TERMINAL, LEAF_SOLVED = 0, 1, 2
UNPROVEN = -128


def _ply(state) -> int:
    return int(state.export_record()[0])


class UctSolveSearch(mcts_spec.Search):
    """mcts_spec.Search with solve=True.  outcome[s] is node s's outcome (Returns() vector) or None."""

    def __init__(self, root, seed: int, tree_stream: int, n_rollouts: int = 1, uct_c: float = 2.0):
        super().__init__(root, seed, tree_stream, n_rollouts, uct_c)
        self.outcome: List[Optional[List[float]]] = [None]

    @property
    def finished(self) -> bool:
        return self.outcome[0] is not None

    def _child_outcome(self, s: int, e: int) -> Optional[List[float]]:
        c = self.nodes[s].children[e]
        return None if c < 0 else self.outcome[c]

    def select(self) -> Tuple[Optional[int], int]:
        """Returns (leaf node index, status); (None, LEAF_SOLVED) once the root is proven."""
        assert self._pending is None
        if self.finished:
            self._pending = ([], None)
            return None, LEAF_SOLVED
        path: List[Tuple[int, int]] = []
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
                e = unvisited[mcts_spec.draw(self.seed, self.T, self.k, len(unvisited))]
            else:
                player = node.state.current_player()
                best, e = None, -1
                for i in range(len(node.actions)):
                    out = self._child_outcome(s, i)
                    sc = (float(out[player]) if out is not None
                          else mcts_spec.uct_score(node.edge_w[i], node.edge_n[i], node.n, self.c))
                    if best is None or sc > best:
                        best, e = sc, i
            path.append((s, e))
            if node.children[e] < 0:
                child = node.state.clone()
                child.apply_action(node.actions[e])
                self.nodes.append(mcts_spec.Node(child, s, node.actions[e]))
                self.outcome.append(None)
                node.children[e] = len(self.nodes) - 1
            s = node.children[e]
        self._pending = (path, s)
        return s, LEAF_TERMINAL if self.nodes[s].state.is_terminal() else LEAF_NEEDS_VALUE

    def backup(self, value: Optional[Sequence[float]] = None) -> None:
        path, leaf = self._pending
        if leaf is None:  # finished tree
            self._pending = None
            self.k += 1
            return
        solved = self.nodes[leaf].state.is_terminal()
        if solved:
            self.outcome[leaf] = [float(x) for x in self.nodes[leaf].state.returns()]
        super().backup(value)
        if not solved:
            return
        for s, _ in reversed(path):
            node = self.nodes[s]
            player = node.state.current_player()
            best, all_solved = None, True
            for c in node.children:
                out = None if c < 0 else self.outcome[c]
                if out is None:
                    all_solved = False
                elif best is None or out[player] > best[player]:
                    best = out
            if best is not None and (all_solved or best[player] == 1.0):
                self.outcome[s] = best
            else:
                break

    # -- results ------------------------------------------------------------------------------------------------
    def root_stats(self, n: int) -> Tuple[np.ndarray, np.ndarray, int]:
        """As twixt_mcts_root_stats of a UCT solver search: best is sort_key's (outcome, N, W), lowest action."""
        visits, sums, _ = super().root_stats(n)
        root = self.nodes[0]
        best = -1
        if root.actions:
            player = root.state.current_player()
            key = lambda i: (0.0 if self._child_outcome(0, i) is None else self._child_outcome(0, i)[player],  # noqa
                             root.edge_n[i], root.edge_w[i])
            bi = 0
            for i in range(len(root.actions)):
                if key(i) > key(bi):
                    bi = i
            best = root.actions[bi]
        return visits, sums, best

    def edge_codes(self, s: int) -> List[int]:
        node = self.nodes[s]
        if node.actions is None:
            return []
        player = node.state.current_player()
        return [0 if self._child_outcome(s, i) is None else 2 + int(self._child_outcome(s, i)[player])
                for i in range(len(node.actions))]

    def solver_stats(self, n: int):
        return _solver_stats(self.outcome[0], _ply(self.nodes[0].state), self.nodes[0].n,
                             [(a, self._child_outcome(0, i)) for i, a in enumerate(self.nodes[0].actions or [])], n)

    def dump(self):
        """Per slot: (parent slot, action, N(s), edge count or -1, [N(a)], [W(a)], [P(a)] (empty), [code])."""
        out = []
        for s, node in enumerate(self.nodes):
            L = -1 if node.actions is None else len(node.actions)
            out.append((node.parent, node.action, node.n, L, list(node.edge_n), list(node.edge_w), None,
                        self.edge_codes(s)))
        return out

    def root_code(self) -> int:
        return 0 if self.outcome[0] is None else 2 + int(self.outcome[0][_ply(self.nodes[0].state) & 1])


class PuctSolveSearch(puct_spec.Search):
    """puct_spec.Search with solve=True (SearchNode.outcome is open_spiel's)."""

    @property
    def finished(self) -> bool:
        return self.nodes[0].outcome is not None

    def select(self) -> Tuple[Optional[int], int]:
        if self.finished:
            assert self._pending is None
            self._pending = "finished"
            return None, LEAF_SOLVED
        leaf, terminal = super().select()
        return leaf, LEAF_TERMINAL if terminal else LEAF_NEEDS_VALUE

    def backup(self, value: Optional[Sequence[float]] = None, priors: Optional[Sequence[float]] = None) -> None:
        if self._pending == "finished":
            self._pending = None
            self.k += 1
            return
        visit_path = list(self._pending)
        solved = visit_path[-1].state.is_terminal()
        super().backup(value, priors)  # sets a terminal leaf's outcome
        if not solved:
            return
        for node in reversed(visit_path):
            if not node.children:
                continue
            player = node.children[0].player
            best, all_solved = None, True
            for child in node.children:
                if child.outcome is None:
                    all_solved = False
                elif best is None or child.outcome[player] > best.outcome[player]:
                    best = child
            if best is not None and (all_solved or best.outcome[player] == 1.0):
                node.outcome = best.outcome
            else:
                break

    def edge_codes(self, node) -> List[int]:
        return [0 if c.outcome is None else 2 + int(c.outcome[c.player]) for c in node.edges()]

    def solver_stats(self, n: int):
        root = self.nodes[0]
        return _solver_stats(root.outcome, _ply(root.state), root.explore_count,
                             [(c.action, c.outcome) for c in root.children], n)

    def dump(self):
        return [d + (self.edge_codes(node),) for d, node in zip(super().dump(), self.nodes)]

    def root_code(self) -> int:
        root = self.nodes[0]
        return 0 if root.outcome is None else 2 + int(root.outcome[_ply(root.state) & 1])


def _solver_stats(root_outcome, root_ply: int, root_visits: int, edges, n: int):
    """(proven, returns [2] float32, edge values [n*n] int8, simulations) as twixt_mcts_solver_stats."""
    values = np.full(n * n, UNPROVEN, dtype=np.int8)
    player = root_ply & 1
    for a, out in edges:
        if out is not None:
            values[a] = int(out[player])
    ret = np.zeros(2, dtype=np.float32) if root_outcome is None else np.asarray(root_outcome, dtype=np.float32)
    return int(root_outcome is not None), ret, values, int(root_visits)


def make(kind: str, root, seed: int, tree_stream: int, n_rollouts: int = 1, uct_c: float = 2.0):
    cls = PuctSolveSearch if kind == "puct" else UctSolveSearch
    return cls(root, seed, tree_stream, n_rollouts, uct_c)


def near_end_roots(game, n: int, seed: int, count: int, back: Sequence[int] = (2, 3, 4, 5)) -> List[object]:
    """Roots `back` plies before the end of seeded fused playouts (cycled), skipping none: the endgames in which
    a solver proves most of its roots."""
    out = []
    for i in range(count):
        st = game.new_initial_state()
        acts = st.clone().playout_philox(seed, 7000 + i)
        b = back[i % len(back)]
        for a in acts[:max(0, len(acts) - b)]:
            st.apply_action(a)
        out.append(st)
    return out


def negamax(state, memo: dict) -> int:
    """Exact value of `state` for its player to move (for a terminal state: for the player whose turn it would be
    by ply parity), memoised on the record bytes."""
    key = state.export_record().tobytes()
    if key in memo:
        return memo[key]
    if state.is_terminal():
        v = int(state.returns()[_ply(state) & 1])
    else:
        v = -1
        for a in state.legal_actions():
            ch = state.clone()
            ch.apply_action(a)
            v = max(v, -negamax(ch, memo))
            if v == 1:
                break
    memo[key] = v
    return v
