"""TEST INFRASTRUCTURE: executable specification of the search with several leaves per step and virtual loss
(include/twixt_b200.h, "Several leaves per step"), written on the UCT and PUCT specifications (mcts_spec,
puct_spec) and so on the oracle alone.

One step is K simulations of every tree.  Every node has a virtual visit count V(s) and every edge V(a), 0 between
steps.  Descent j = 0 .. K-1 of a step is simulation k = self.k + j (the k of the unvisited-edge draw and of the
rollout streams) and scores with n_eff = N(a) + V(a), N_eff(s) = N(s) + V(s) and
w_eff = (V(a) > 0 ? W(a) - vl * V(a) : W(a)); after it picks its path, V += 1 on every edge and node of the path and
on the leaf.  The leaf rule is unchanged (a terminal node or N(s) == 0).  `backup_step` takes rows j = 0 .. K-1 in
order: row j removes its virtual visits and backs up as the base search does; a PUCT leaf is expanded by the lowest
row whose leaf it is.  K = 1 is the base search exactly.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import mcts_spec
import puct_spec


def w_eff(w: float, v: int, vl: float) -> float:
    return w - vl * v if v > 0 else w


class UctSearch(mcts_spec.Search):
    """mcts_spec.Search with K descents per step.  self.vn[s] is V(s), self.ve[s][i] V(a) of edge i of node s."""

    def __init__(self, root, seed: int, tree_stream: int, n_rollouts: int = 1, uct_c: float = 2.0,
                 virtual_loss: float = 1.0):
        super().__init__(root, seed, tree_stream, n_rollouts, uct_c)
        self.vl = float(virtual_loss)
        self.vn: List[int] = [0]
        self.ve: List[List[int]] = [[]]
        self._rows: Optional[List[Tuple[List[Tuple[int, int]], int]]] = None

    def _descend(self, k: int) -> Tuple[List[Tuple[int, int]], int]:
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
                self.ve[s] = [0] * L
            ve = self.ve[s]
            unvisited = [i for i, v in enumerate(node.edge_n) if v + ve[i] == 0]
            if unvisited:
                e = unvisited[mcts_spec.draw(self.seed, self.T, k, len(unvisited))]
            else:
                best, e = None, -1
                for i in range(len(node.actions)):
                    sc = mcts_spec.uct_score(w_eff(node.edge_w[i], ve[i], self.vl), node.edge_n[i] + ve[i],
                                             node.n + self.vn[s], self.c)
                    if best is None or sc > best:
                        best, e = sc, i
            path.append((s, e))
            if node.children[e] < 0:
                child = node.state.clone()
                child.apply_action(node.actions[e])
                self.nodes.append(mcts_spec.Node(child, s, node.actions[e]))
                self.vn.append(0)
                self.ve.append([])
                node.children[e] = len(self.nodes) - 1
            s = node.children[e]
        for p, e in path:
            self.vn[p] += 1
            self.ve[p][e] += 1
        self.vn[s] += 1
        return path, s

    def select_step(self, K: int) -> List[Tuple[int, bool]]:
        """K descents; returns [(leaf node, leaf is terminal)] by row j."""
        assert self._rows is None and self._pending is None
        self._rows = [self._descend(self.k + j) for j in range(K)]
        return [(leaf, self.nodes[leaf].state.is_terminal()) for _, leaf in self._rows]

    def backup_step(self, values: Sequence[Optional[Sequence[float]]], priors=None) -> None:
        """values[j]: row j's [2] values (ignored for a terminal leaf).  UCT takes no priors."""
        rows, self._rows = self._rows, None
        for (path, leaf), value in zip(rows, values):
            for p, e in path:
                self.vn[p] -= 1
                self.ve[p][e] -= 1
            self.vn[leaf] -= 1
            self._pending = (path, leaf)
            self.backup(value)  # N, W and self.k += 1 as the base search

    def rollout_value_at(self, leaf: int, k: int) -> List[float]:
        saved, self.k = self.k, k
        try:
            return self.rollout_value(leaf)
        finally:
            self.k = saved

    def run_steps(self, num_simulations: int, K: int, value_fn=None) -> "UctSearch":
        assert num_simulations % K == 0
        for _ in range(num_simulations // K):
            leaves = self.select_step(K)
            vals = []
            for j, (leaf, terminal) in enumerate(leaves):
                if terminal:
                    vals.append(None)
                elif value_fn is None:
                    vals.append(self.rollout_value_at(leaf, self.k + j))
                else:
                    vals.append(value_fn(self.nodes[leaf].state.export_record()))
            self.backup_step(vals)
        return self

    def virtual_counts(self) -> List[int]:
        return self.vn + [v for ve in self.ve for v in ve]


class PuctSearch(puct_spec.Search):
    """puct_spec.Search with K descents per step.  self.v[slot] is V of that node and of the edge into it."""

    def __init__(self, root, seed: int, tree_stream: int, n_rollouts: int = 1, uct_c: float = 2.0,
                 virtual_loss: float = 1.0):
        super().__init__(root, seed, tree_stream, n_rollouts, uct_c)
        self.vl = float(virtual_loss)
        self.v: List[int] = [0]
        self._rows = None

    def _score(self, child, parent_eff: int) -> float:
        # an edge whose child exists and is terminal scores its outcome, also before its first backup (a child
        # an earlier descent of the same step created)
        if child.outcome is not None:
            return child.outcome[child.player]
        if child.slot is not None and child.state.is_terminal():
            return float(child.state.returns()[child.player])
        v = self.v[child.slot] if child.slot is not None else 0
        n = child.explore_count + v
        w = w_eff(child.total_reward, v, self.vl)
        return (n and w / n) + self.c * child.prior * math.sqrt(parent_eff) / (n + 1)

    def _descend(self):
        current = self.nodes[0]
        visit_path = [current]
        while not current.state.is_terminal() and current.explore_count > 0:
            parent_eff = current.explore_count + self.v[current.slot]
            chosen = max(current.children, key=lambda c: self._score(c, parent_eff))
            if chosen.slot is None:
                chosen.state = current.state.clone()
                chosen.state.apply_action(chosen.action)
                chosen.slot = len(self.nodes)
                chosen.parent_slot = current.slot
                self.nodes.append(chosen)
                self.v.append(0)
            current = chosen
            visit_path.append(current)
        for node in visit_path:
            self.v[node.slot] += 1
        return visit_path

    def select_step(self, K: int) -> List[Tuple[int, bool]]:
        assert self._rows is None and self._pending is None
        self._rows = [self._descend() for _ in range(K)]
        return [(p[-1].slot, p[-1].state.is_terminal()) for p in self._rows]

    def backup_step(self, values, priors=None) -> None:
        """values[j] / priors[j]: row j's [2] values and [n*n] priors (None: uniform); ignored for a terminal
        leaf, and the priors also for a leaf an earlier row of the step expanded."""
        rows, self._rows = self._rows, None
        expanded = set()
        for j, visit_path in enumerate(rows):
            leaf = visit_path[-1]
            for node in visit_path:
                self.v[node.slot] -= 1
            repeated = leaf.slot in expanded
            expanded.add(leaf.slot)
            self._pending = visit_path
            if repeated:
                kids = leaf.children
                self.backup(values[j], None)  # expands the leaf again: put back the first row's children
                leaf.children = kids
            else:
                self.backup(values[j], None if priors is None else priors[j])

    def rollout_value_at(self, leaf: int, k: int) -> List[float]:
        saved, self.k = self.k, k
        try:
            return self.rollout_value(leaf)
        finally:
            self.k = saved

    def run_steps(self, num_simulations: int, K: int, value_fn=None, prior_fn=None) -> "PuctSearch":
        assert num_simulations % K == 0
        for _ in range(num_simulations // K):
            leaves = self.select_step(K)
            vals, pri = [], []
            for j, (leaf, terminal) in enumerate(leaves):
                rec = self.nodes[leaf].state.export_record()
                if terminal:
                    vals.append(None)
                elif value_fn is None:
                    vals.append(self.rollout_value_at(leaf, self.k + j))
                else:
                    vals.append(value_fn(rec))
                pri.append(None if (terminal or prior_fn is None) else prior_fn(rec))
            self.backup_step(vals, pri)
        return self

    def virtual_counts(self) -> List[int]:
        return list(self.v)
