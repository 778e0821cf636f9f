"""TEST INFRASTRUCTURE: executable specification of the Gumbel AlphaZero search (include/twixt_b200.h, "Gumbel
AlphaZero search"), written on the oracle (oracle/pyoracle.py) and tests/puct_spec.py, and nothing else.

It restates DeepMind mctx's gumbel_muzero_policy (policies.py), seq_halving.py (score_considered,
get_sequence_of_considered_visits, get_table_of_considered_visits), qtransforms.qtransform_completed_by_mix_value
(with its defaults: rescale_values, use_mixed_value, epsilon = 1e-8; _compute_mixed_value, _complete_qvalues,
_rescale_qvalues) and action_selection.gumbel_muzero_root_action_selection / gumbel_muzero_interior_action_selection,
with the substitutions that make it reproducible on the GPU:
  * IEEE double arithmetic in plain Python floats instead of float32 JAX; logits and noise are stored as float32;
  * every exp is `mcts_exp` below (twixt_mcts.cuh's, line for line) and every sum over a node's edges is `warp_sum`
    (lane l adds edges l, l+32, .. from 0.0, then an xor butterfly over offsets 16, 8, 4, 2, 1);
  * the tree is the PUCT search's (puct_spec.Search): one node per simulation in creation order, a leaf at a
    terminal node or one with N(s) = 0, expanded at its backup with the caller's logits (0 without), edges the
    legal actions ascending.  The root's own evaluation is simulation 0, so the root's Sequential Halving index is
    sum N(a) = N(root) - 1 and its table has max_simulations - 1 columns.
Node values: W(a) is summed for the player to move at the parent, as in PUCT; v(s) is the evaluation of s for the
player to move at s (ply parity).
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence

import numpy as np

import puct_spec
from puct_spec import SearchNode, f32

TINY = float.fromhex("0x1.0p-1022")  # the smallest normal double (mctx: jnp.finfo(dtype).tiny)
EPSILON = 1e-8
LOW_LOGIT = -1e9
LOG2E = float.fromhex("0x1.71547652b82fep+0")
LN2_HI = float.fromhex("0x1.62e42fee00000p-1")
LN2_LO = float.fromhex("0x1.a39ef35793c76p-33")
# float64(1/j!), j = 13 .. 0, in Horner order
EXP_COEFFS = [float.fromhex(h) for h in (
    "0x1.6124613a86d09p-33", "0x1.1eed8eff8d898p-29", "0x1.ae64567f544e4p-26", "0x1.27e4fb7789f5cp-22",
    "0x1.71de3a556c734p-19", "0x1.a01a01a01a01ap-16", "0x1.a01a01a01a01ap-13", "0x1.6c16c16c16c17p-10",
    "0x1.1111111111111p-7", "0x1.5555555555555p-5", "0x1.5555555555555p-3", "0x1.0p-1", "0x1.0p+0", "0x1.0p+0")]


def mcts_exp(x: float) -> float:
    """twixt_mcts.cuh mcts_exp: exp(x) for x <= 0."""
    if not x >= -746.0:
        return 0.0
    k = round(x * LOG2E)  # round half to even
    r = (x - k * LN2_HI) - k * LN2_LO
    p = EXP_COEFFS[0]
    for c in EXP_COEFFS[1:]:
        p = p * r + c
    return (p * math.ldexp(1.0, k >> 1)) * math.ldexp(1.0, k - (k >> 1))


def warp_sum(L: int, term, include=None) -> float:
    """The device's order of a sum over L edges: term(i) for the edges with include(i)."""
    p = [0.0] * 32
    for lane in range(32):
        for i in range(lane, L, 32):
            if include is None or include(i):
                p[lane] = p[lane] + term(i)
    for d in (16, 8, 4, 2, 1):
        p = [p[lane] + p[lane ^ d] for lane in range(32)]
    return p[0]


def considered_visits(m: int, num_simulations: int) -> List[int]:
    """mctx get_sequence_of_considered_visits(m, num_simulations) in integer arithmetic."""
    if m <= 1:
        return list(range(num_simulations))
    log2max = (m - 1).bit_length()  # ceil(log2(m))
    sequence: List[int] = []
    visits = [0] * m
    num_considered = m
    while len(sequence) < num_simulations:
        extra = max(1, num_simulations // (log2max * num_considered))
        for _ in range(extra):
            sequence.extend(visits[:num_considered])
            for i in range(num_considered):
                visits[i] += 1
        num_considered = max(2, num_considered // 2)
    return sequence[:num_simulations]


def considered_table(max_considered: int, num_simulations: int) -> List[List[int]]:
    """mctx get_table_of_considered_visits."""
    return [considered_visits(m, num_simulations) for m in range(max_considered + 1)]


def completed_q(logits: Sequence[float], visits: Sequence[int], sums: Sequence[float], raw_value: float,
                c_visit: float, c_scale: float) -> dict:
    """qtransform_completed_by_mix_value at one node from its edges' l, N, W and its v: returns the pieces
    (max_logit, pi, sum_n, v_mix, q_completed, sigma)."""
    L = len(logits)
    mx = max(logits)
    sum_n = sum(visits)
    max_n = max(visits)
    z = warp_sum(L, lambda i: mcts_exp(logits[i] - mx))
    pi = [max(mcts_exp(logits[i] - mx) / z, TINY) for i in range(L)]
    weighted_q = 0.0
    if sum_n > 0:
        visited = lambda i: visits[i] > 0  # noqa: E731
        sum_probs = warp_sum(L, lambda i: pi[i], visited)
        weighted_q = warp_sum(L, lambda i: (pi[i] * (sums[i] / visits[i])) / sum_probs, visited)
    v_mix = (raw_value + float(sum_n) * weighted_q) / (float(sum_n) + 1.0)
    q = [sums[i] / visits[i] if visits[i] > 0 else v_mix for i in range(L)]
    q_min, q_max = min(q), max(q)
    scale = (c_visit + float(max_n)) * c_scale
    sigma = [scale * ((x - q_min) / max(q_max - q_min, EPSILON)) for x in q]
    return {"max_logit": mx, "pi": pi, "sum_n": sum_n, "max_n": max_n, "v_mix": v_mix, "q": q, "sigma": sigma}


def improved_policy(logits: Sequence[float], sigma: Sequence[float]) -> List[float]:
    """softmax(l + sigma) in the device's order (the interior rule's pi' and the root's action weights)."""
    x = [logits[i] + sigma[i] for i in range(len(logits))]
    mx = max(x)
    z = warp_sum(len(x), lambda i: mcts_exp(x[i] - mx))
    return [mcts_exp(v - mx) / z for v in x]


def argmax(scores: Sequence[Optional[float]]) -> int:
    """The first index of the largest score (jnp.argmax); None entries are not eligible; -1 if none is."""
    best, bi = None, -1
    for i, s in enumerate(scores):
        if s is not None and (best is None or s > best):
            best, bi = s, i
    return bi


def root_scores(cq: dict, logits, noise, visits, considered: int) -> List[Optional[float]]:
    """seq_halving.score_considered: max(-1e9, (g + (l - max l)) + sigma) on the edges with N = considered."""
    return [max(LOW_LOGIT, (noise[i] + (logits[i] - cq["max_logit"])) + cq["sigma"][i]) if visits[i] == considered
            else None for i in range(len(logits))]


def ply_parity(state) -> int:
    return int(state.export_record()[0]) & 1


class GNode(SearchNode):
    """A PUCT SearchNode with its logit l (float32) and, once evaluated, its raw value v."""
    __slots__ = ("logit", "raw_value")

    def __init__(self, action, player, logit=0.0, edge=-1):
        super().__init__(action, player, 0.0, edge, 0)
        self.logit = logit
        self.raw_value = 0.0


class Search(puct_spec.Search):
    """One Gumbel tree.  `root` is an OracleState (copied); `gumbel` the root noise [n*n] (None: 0)."""

    def __init__(self, root, seed: int, tree_stream: int, n_rollouts: int = 1, max_simulations: int = 16,
                 max_considered: int = 16, c_visit: float = 50.0, c_scale: float = 0.1, gumbel=None):
        super().__init__(root, seed, tree_stream, n_rollouts)
        r = GNode(None, max(root.current_player(), 0))
        r.slot, r.state = 0, root.clone()
        self.nodes = [r]
        self.max_considered = int(max_considered)
        self.c_visit = float(c_visit)
        self.c_scale = float(c_scale)
        self.table = considered_table(self.max_considered, max_simulations - 1)
        self.set_root_gumbel(gumbel)

    def set_root_gumbel(self, gumbel) -> None:
        self.gumbel = None if gumbel is None else [float(x) for x in np.asarray(gumbel, dtype=np.float32)]

    def _node_q(self, node) -> dict:
        e = node.edges()
        return completed_q([c.logit for c in e], [c.explore_count for c in e], [c.total_reward for c in e],
                           node.raw_value, self.c_visit, self.c_scale)

    def _root_noise(self, edges) -> List[float]:
        return [0.0 if self.gumbel is None else self.gumbel[c.action] for c in edges]

    def _root_edge(self, node) -> int:
        e = node.edges()
        cq = self._node_q(node)
        m = min(self.max_considered, len(e))
        visits = [c.explore_count for c in e]
        considered = self.table[m][cq["sum_n"]]
        i = argmax(root_scores(cq, [c.logit for c in e], self._root_noise(e), visits, considered))
        return 0 if i < 0 else i

    def _interior_edge(self, node) -> int:
        e = node.edges()
        cq = self._node_q(node)
        pi2 = improved_policy([c.logit for c in e], cq["sigma"])
        sn = float(cq["sum_n"])
        return argmax([pi2[i] - float(c.explore_count) / (sn + 1.0) for i, c in enumerate(e)])

    # -- descent: the root by Sequential Halving, other nodes by the interior rule -------------------------------
    def select(self):
        assert self._pending is None
        current = self.nodes[0]
        visit_path = [current]
        while not current.state.is_terminal() and current.explore_count > 0:
            i = self._root_edge(current) if current.slot == 0 else self._interior_edge(current)
            chosen = current.edges()[i]
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

    # -- backup, v(leaf), and the expansion of a non-terminal leaf with its logits --------------------------------
    def backup(self, value=None, logits=None) -> None:
        visit_path = self._pending
        leaf = visit_path[-1]
        st = leaf.state
        if st.is_terminal():
            returns = [float(x) for x in st.returns()]
        else:
            returns = [float(value[0]), float(value[1])]
        for node in visit_path:
            node.total_reward += returns[node.player]
            node.explore_count += 1
        leaf.raw_value = returns[ply_parity(st)]
        if not st.is_terminal():
            player = st.current_player()
            leaf.children = [GNode(a, player, 0.0 if logits is None else f32(logits[a]), i)
                             for i, a in enumerate(st.legal_actions())]
        self._pending = None
        self.k += 1

    # -- results ------------------------------------------------------------------------------------------------
    def gumbel_stats(self, n: int):
        """(action or -1, improved policy [n*n] float32) as twixt_mcts_gumbel_stats."""
        root = self.nodes[0]
        policy = np.zeros(n * n, dtype=np.float32)
        if not root.children:
            return -1, policy
        e = root.edges()
        cq = self._node_q(root)
        logits = [c.logit for c in e]
        visits = [c.explore_count for c in e]
        action = e[argmax(root_scores(cq, logits, self._root_noise(e), visits, cq["max_n"]))].action
        for c, p in zip(e, improved_policy(logits, cq["sigma"])):
            policy[c.action] = np.float32(p)
        return action, policy

    def root_stats(self, n: int):
        """(visits, value_sums, Gumbel action) as twixt_mcts_root_stats on a Gumbel search."""
        visits = np.zeros(n * n, dtype=np.int32)
        sums = np.zeros(n * n, dtype=np.float64)
        for c in self.nodes[0].children:
            visits[c.action] = c.explore_count
            sums[c.action] = c.total_reward
        return visits, sums, self.gumbel_stats(n)[0]

    def dump(self):
        """Per slot: (parent slot, action, N(s), edge count or -1, [N(a)], [W(a)], [l(a)], v) in edge order."""
        out = []
        for node in self.nodes:
            e = node.edges()
            L = len(e) if node.children else -1
            out.append((node.parent_slot, -1 if node.action is None else node.action, node.explore_count, L,
                        [c.explore_count for c in e], [c.total_reward for c in e], [c.logit for c in e],
                        node.raw_value))
        return out


def stand_in_logits(record: np.ndarray, n: int) -> np.ndarray:
    """Deterministic float32 logits [n*n] of a leaf record for the stepwise tests: log of puct_spec's stand-in
    priors (-inf where they are 0, which includes illegal cells the search must ignore) plus a hashed offset, so that
    rows differ in scale as a network's logits do."""
    p = puct_spec.stand_in_priors(record, n).astype(np.float64)
    h = int(np.bitwise_xor.reduce(record.astype(np.uint64) * np.uint64(0x27D4EB2F)))
    with np.errstate(divide="ignore"):
        out = np.log(p) * (0.5 + (h & 7) / 4.0) + ((h >> 3) & 15) - 7.0
    return out.astype(np.float32)
