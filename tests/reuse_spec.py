"""TEST INFRASTRUCTURE: executable specification of tree reuse across moves (include/twixt_b200.h,
twixt_mcts_advance), written on the UCT, PUCT, solver and virtual-loss specifications (mcts_spec, puct_spec,
solver_spec, vl_spec) and so on the oracle alone.

`advance(search, action, keep_nodes)` moves a specification search's root along `action`:
  * a legal action whose root edge has a child: the kept nodes are that child's subtree, renumbered by their rank in
    old slot order (the new root is slot 0, children stay above their parents), and only the first keep_nodes of
    that order are kept.  Every kept node keeps all its statistics; an edge whose child the cap drops is unvisited
    again (N = 0, W = 0, no child) but keeps its prior, tie key and outcome;
  * a legal action without a child: the tree is cleared to the root with the move applied, as begin would;
  * -1: the root stays and only the cap applies;
  * an illegal action (anything but -1 at a terminal root included): nothing changes, status ROOT_ILLEGAL.
A solver search's new root takes the outcome of the chosen edge's child (proven or terminal), also when the cap
dropped that child earlier.  The simulation counter k carries on.

The UCT specifications keep a child's outcome on the child node; an edge whose proven child the cap dropped keeps
that outcome as its code on the device, so the UCT solver class below keeps it per edge (`ghost`) until the child
is created again.  The PUCT specifications keep it on the SearchNode, which the reset leaves in its parent's list.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import mcts_spec
import puct_spec
import solver_spec
import vl_spec

ROOT_KEPT, ROOT_ILLEGAL, ROOT_FRESH = 0, 1, 2


def _legal(state, action: int) -> bool:
    return not state.is_terminal() and action in state.legal_actions()


# ------------------------------------------------------------------------------------------------------- UCT ---
class UctSolveSearch(solver_spec.UctSolveSearch):
    """solver_spec.UctSolveSearch whose edges keep the outcome of a child the cap dropped (ghost[(slot, edge)]),
    as the device keeps the edge's code: selection, proofs and results read it until the child is created again,
    which then takes it as its outcome."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.ghost: Dict[Tuple[int, int], List[float]] = {}

    def _child_outcome(self, s: int, e: int) -> Optional[List[float]]:
        c = self.nodes[s].children[e]
        return self.ghost.get((s, e)) if c < 0 else self.outcome[c]

    def select(self):
        assert self._pending is None
        if self.finished:
            self._pending = ([], None)
            return None, solver_spec.LEAF_SOLVED
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
                self.outcome.append(self.ghost.pop((s, e), None))
                node.children[e] = len(self.nodes) - 1
            s = node.children[e]
        self._pending = (path, s)
        return s, solver_spec.LEAF_TERMINAL if self.nodes[s].state.is_terminal() else solver_spec.LEAF_NEEDS_VALUE

    def backup(self, value: Optional[Sequence[float]] = None) -> None:
        path, leaf = self._pending
        if leaf is None:
            self._pending = None
            self.k += 1
            return
        solved = self.nodes[leaf].state.is_terminal()
        if solved:
            self.outcome[leaf] = [float(x) for x in self.nodes[leaf].state.returns()]
        mcts_spec.Search.backup(self, value)
        if not solved:
            return
        for s, _ in reversed(path):
            node = self.nodes[s]
            player = node.state.current_player()
            best, all_solved = None, True
            for i in range(len(node.children)):
                out = self._child_outcome(s, i)
                if out is None:
                    all_solved = False
                elif best is None or out[player] > best[player]:
                    best = out
            if best is not None and (all_solved or best[player] == 1.0):
                self.outcome[s] = best
            else:
                break


def _uct_advance(s, action: int, keep: int) -> int:
    solve = isinstance(s, solver_spec.UctSolveSearch)
    if solve:
        assert isinstance(s, UctSolveSearch), "use reuse_spec.UctSolveSearch: it keeps the codes of dropped edges"
    virtual = isinstance(s, vl_spec.UctSearch)
    root = s.nodes[0]
    start = 0
    if action != -1:
        if not _legal(root.state, action):
            return ROOT_ILLEGAL
        child, outcome = -1, None
        if root.actions is not None:
            e = root.actions.index(action)
            child = root.children[e]
            if solve:
                outcome = s._child_outcome(0, e)
        if child < 0:
            st = root.state.clone()
            st.apply_action(action)
            s.nodes = [mcts_spec.Node(st, -1, -1)]
            if solve:
                s.outcome = [outcome]
                s.ghost = {}
            if virtual:
                s.vn, s.ve = [0], [[]]
            return ROOT_FRESH
        start = child
    # the subtree of `start` in slot order: a slot is in it when a kept parent (a lower slot) reaches it
    reached, order = {start}, []
    for sl in range(start, len(s.nodes)):
        if len(order) == keep:
            break
        if sl in reached:
            order.append(sl)
            reached.update(c for c in s.nodes[sl].children if c >= 0)
    new = {old: i for i, old in enumerate(order)}
    nodes, outcome, ghost = [], [], {}
    for old in order:
        nd = s.nodes[old]
        nd.parent, nd.action = (-1, -1) if old == start else (new[nd.parent], nd.action)
        for i, c in enumerate(nd.children):
            if c >= 0 and c not in new:  # dropped by the cap: unvisited again
                nd.edge_n[i], nd.edge_w[i], nd.children[i] = 0, 0.0, -1
                if solve and s.outcome[c] is not None:
                    ghost[(new[old], i)] = s.outcome[c]
            elif c >= 0:
                nd.children[i] = new[c]
            elif solve and (old, i) in s.ghost:
                ghost[(new[old], i)] = s.ghost[(old, i)]
        nodes.append(nd)
        if solve:
            outcome.append(s.outcome[old])
    s.nodes = nodes
    if solve:
        s.outcome, s.ghost = outcome, ghost
    if virtual:
        s.vn = [0] * len(nodes)
        s.ve = [[0] * len(nd.edge_n) for nd in nodes]
    return ROOT_KEPT if s.nodes[0].n > 0 else ROOT_FRESH


# ------------------------------------------------------------------------------------------------------ PUCT ---
def _reset(node: puct_spec.SearchNode) -> None:
    """A child the cap dropped: a fresh node; its action, player, prior, edge, tie key and outcome stay."""
    node.slot, node.state, node.children = None, None, []
    node.explore_count, node.total_reward = 0, 0.0
    node.parent_slot = -1


def _puct_advance(s, action: int, keep: int) -> int:
    solve = isinstance(s, solver_spec.PuctSolveSearch)
    virtual = isinstance(s, vl_spec.PuctSearch)
    root = s.nodes[0]
    start = root
    if action != -1:
        if not _legal(root.state, action):
            return ROOT_ILLEGAL
        edge = next((c for c in root.children if c.action == action), None)
        if edge is None or edge.slot is None:
            st = root.state.clone()
            st.apply_action(action)
            r = puct_spec.SearchNode(None, max(st.current_player(), 0), 1.0)
            r.slot, r.state = 0, st
            if solve and edge is not None:
                r.outcome = edge.outcome
            s.nodes = [r]
            if virtual:
                s.v = [0]
            return ROOT_FRESH
        start = edge
    reached, order = {start.slot}, []
    for sl in range(start.slot, len(s.nodes)):
        if len(order) == keep:
            break
        if sl in reached:
            order.append(s.nodes[sl])
            reached.update(c.slot for c in s.nodes[sl].children if c.slot is not None)
    new = {nd.slot: i for i, nd in enumerate(order)}
    for nd in order:
        for c in nd.children:
            if c.slot is not None and c.slot not in new:
                _reset(c)
    for nd in order:
        nd.parent_slot = -1 if nd is start else new[nd.parent_slot]
        nd.slot = new[nd.slot]
    if start is not root:
        start.action = None
    s.nodes = order
    if virtual:
        s.v = [0] * len(order)
    return ROOT_KEPT if start.explore_count > 0 else ROOT_FRESH


def advance(search, action: int, keep_nodes: int) -> int:
    """twixt_mcts_advance of one tree on a specification search (any of mcts_spec.Search, puct_spec.Search, their
    solver classes -- reuse_spec.UctSolveSearch for UCT -- and the virtual-loss classes); returns its status."""
    assert keep_nodes >= 1
    assert search._pending is None and getattr(search, "_rows", None) is None
    if isinstance(search, puct_spec.Search):
        return _puct_advance(search, int(action), int(keep_nodes))
    return _uct_advance(search, int(action), int(keep_nodes))


def make(kind: str, root, seed: int, tree_stream: int, n_rollouts: int = 1, uct_c: float = 2.0, solve: bool = False,
         K: int = 1, virtual_loss: float = 1.0):
    """A specification search of the device kind (selection "uct" / "puct", solve, leaves_per_step K)."""
    assert not (solve and K > 1)
    if solve:
        cls = UctSolveSearch if kind == "uct" else solver_spec.PuctSolveSearch
        return cls(root, seed, tree_stream, n_rollouts, uct_c)
    if K > 1:
        cls = vl_spec.UctSearch if kind == "uct" else vl_spec.PuctSearch
        return cls(root, seed, tree_stream, n_rollouts, uct_c, virtual_loss)
    cls = mcts_spec.Search if kind == "uct" else puct_spec.Search
    return cls(root, seed, tree_stream, n_rollouts, uct_c)


def node_count(search) -> int:
    return len(search.nodes)


def check_tree(search) -> None:
    """Structural invariants: slots number the nodes, every child slot is above its parent's, every node but the
    root is reached from exactly one edge, and N(s) of an expanded node is at least the sum of its edges' N."""
    if isinstance(search, puct_spec.Search):
        seen = {0}
        for i, nd in enumerate(search.nodes):
            assert nd.slot == i
            for c in nd.children:
                if c.slot is not None:
                    assert c.slot > i and c.parent_slot == i and c.slot not in seen
                    seen.add(c.slot)
            assert nd.explore_count >= sum(c.explore_count for c in nd.children) or i == 0
    else:
        seen = {0}
        for i, nd in enumerate(search.nodes):
            for c in nd.children:
                if c >= 0:
                    assert c > i and search.nodes[c].parent == i and c not in seen
                    seen.add(c)
            if nd.actions is not None:
                assert nd.n >= sum(nd.edge_n)
    assert seen == set(range(len(search.nodes)))
