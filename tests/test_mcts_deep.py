"""Batched MCTS on deep trees and past one warp of rollouts and leaves.

The device kernels (twixt_mcts.cu) work with one warp per tree, and several of their loops stride over a tree's path,
its rollout slots or its leaf rows 32 lanes at a time: the N / W updates of the backups, the virtual-visit adds and
removals, the solver's proof walk, the advance's subtree walk and the rollout-id loops of the select kernels.  The
searches the other MCTS tests run are a few nodes deep with R <= 8 rollouts per leaf, so none of those loops takes a
second lane pass there.  Here every search kind is driven down a *line*: priors, logits or values that make each
simulation extend one chain of the tree by a node, to depths of 33 .. 600 (a whole game at n = 24), and R, K and
K * R go past 32.

A line's move at a node is a hash of the node's record over its legal actions (`line_action`).  Every test asserts
what its specification trees reach (depth, terminal nodes inside the tree, node count), so that an edit that makes a
recipe shallow fails here instead of silently testing less.

CPU: the host-compiled harnesses node for node against the specifications on the deep recipes.  GPU: the device
search bit for bit against the specifications (leaf records and statuses at every step, root, solver and Gumbel
stats, advance statuses, twixt_stats), plus checks that do not rest on the specifications: the PUCT line's leaves,
root visits and root value sum from the oracle alone, and the Gumbel line's improved policy from a float64 softmax."""
import numpy as np
import pytest

import gumbel_spec
import mcts_spec
import puct_spec
import reuse_spec
import solver_spec
import test_mcts_gumbel as tg
import test_mcts_puct as tp
import test_mcts_reuse as tr
import test_mcts_solver as ts
import test_mcts_virtual_loss as tv
import vl_spec
from test_mcts_gumbel import gh  # noqa: F401  (fixtures: the host harnesses)
from test_mcts_puct import ph  # noqa: F401
from test_mcts_solver import sh  # noqa: F401
from test_mcts_virtual_loss import vh  # noqa: F401

P = tp.P
M64 = (1 << 64) - 1
ONES = np.ones(2, dtype=np.float32)  # the UCT line's value: every visited edge ties at c = 0


# ------------------------------------------------------------------------------------------------ lines ---
def line_action(state) -> int:
    """The line's move at a non-terminal state: a hash of its record picks one of its legal actions."""
    legal = state.legal_actions()
    rec = state.export_record().astype(np.uint64)
    h = int(np.bitwise_xor.reduce(rec * np.uint64(0x9E3779B97F4A7C15) + np.arange(rec.size, dtype=np.uint64)))
    h = ((h ^ (h >> 31)) * 0xBF58476D1CE4E5B9) & M64
    h ^= h >> 29
    return legal[h % len(legal)]


def line_priors(state, n: int) -> np.ndarray:
    """Weight 1 on the line's move and 1e-6 on every other legal action, normalised (float32 [n*n])."""
    p = np.zeros(n * n, dtype=np.float64)
    p[state.legal_actions()] = 1e-6
    p[line_action(state)] = 1.0
    return (p / p.sum()).astype(np.float32)


def line_logits(state, n: int, spread: bool = False) -> np.ndarray:
    """+20 on the line's move, 0 elsewhere; spread: the other cells get hashed logits in [0, 1.5] instead."""
    out = np.zeros(n * n, dtype=np.float32)
    if spread:
        rec = state.export_record().astype(np.uint64)
        h = int(np.bitwise_xor.reduce(rec * np.uint64(0x27D4EB2F))) & 0xFFFFFFFF
        out[:] = (((np.arange(n * n) * 0x85EBCA6B + h) >> 5) % 7) / 4.0
    out[line_action(state)] = 20.0
    return out


class Evaluator:
    """value and prior (or logit) rows of a leaf state, remembered by record so that a harness, which only sees the
    record, is answered exactly as the specification was.  A record the specification never evaluated is a
    KeyError: the harness reached a leaf the specification did not."""

    def __init__(self, n, kind):
        self.n, self.kind = n, kind
        self.memo = {}

    def __call__(self, state):
        rec = state.export_record()
        key = rec.tobytes()
        if key not in self.memo:
            n = self.n
            if self.kind == "uct":
                self.memo[key] = (ONES, None)
            elif self.kind == "puct":
                self.memo[key] = (mcts_spec.stand_in_value(rec), line_priors(state, n))
            else:  # "gumbel" / "gumbel-spread"
                self.memo[key] = (mcts_spec.stand_in_value(rec), line_logits(state, n, self.kind == "gumbel-spread"))
        return self.memo[key]

    def value(self, rec):
        return self.memo[rec.tobytes()][0]

    def prior(self, rec):
        return self.memo[rec.tobytes()][1]


def _is_puct_family(ref) -> bool:
    return isinstance(ref, puct_spec.Search)  # PUCT, its solver, virtual-loss and Gumbel classes


def drive(ref, sims, ev):
    """sims simulations of a K = 1 specification search with the evaluator; returns the statuses."""
    statuses = []
    for _ in range(sims):
        leaf, st = ref.select()
        statuses.append(int(st))
        args = (None, None) if _is_puct_family(ref) else (None,)
        if not st:
            v, p = ev(ref.nodes[leaf].state)
            args = (v, p) if _is_puct_family(ref) else (v,)
        ref.backup(*args)
    return statuses


def reach(ref):
    """(maximum depth, terminal nodes below the root, node count) of a specification tree."""
    depth = [0] * len(ref.nodes)
    terminals = 0
    for i, nd in enumerate(ref.nodes):
        if i:
            depth[i] = depth[nd.parent_slot if _is_puct_family(ref) else nd.parent] + 1
            terminals += bool(nd.state.is_terminal())
    return max(depth), terminals, len(ref.nodes)


def oracle_line(root, length):
    """The line followed from the root on the oracle alone: [state after the first k moves for k = 0 ..] until
    length + 1 states or a terminal one."""
    out = [root.clone()]
    while len(out) <= length and not out[-1].is_terminal():
        st = out[-1].clone()
        st.apply_action(line_action(st))
        out.append(st)
    return out


def check_puct_line_root(root, n, sims, visits, sums):
    """The PUCT line without the specification: simulation k's leaf is the line's state after min(k, end) moves,
    so the root's line edge has all sims - 1 visits, every other edge none, and its value sum is the leaf values in
    simulation order (stand-in values, the terminal's returns once the line ends in a win), added in float64.
    Returns False, checking nothing, where the line ends in a draw (the search branches off above a draw)."""
    line = oracle_line(root, sims)
    end = line[-1]
    if end.is_terminal() and max(end.returns()) == 0.0:
        return False
    player = root.current_player()
    w = 0.0
    for k in range(1, sims):
        st = line[min(k, len(line) - 1)]
        v = st.returns() if st.is_terminal() else mcts_spec.stand_in_value(st.export_record())
        w += float(v[player])
    a = line_action(root)
    want = np.zeros(n * n, dtype=np.int32)
    want[a] = sims - 1
    assert np.array_equal(visits, want)
    assert sums[a] == w and not np.any(np.delete(sums, a))
    return True


def assert_uct_line_reach(refs, n):
    reached = [reach(ref) for ref in refs]
    if n >= 8:  # one new node per simulation
        assert max(d for d, _, _ in reached) >= 33 and all(c == ref.k for (_, _, c), ref in zip(reached, refs)), reached
    else:
        assert min(d for d, _, _ in reached) >= 10 and all(t >= 1 for _, t, _ in reached), reached


def line_roots(game, count, seed):
    """Roots for deep lines: the initial position, then positions 1, 2, 3, .. random moves in."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(count):
        st = game.new_initial_state()
        for _ in range(i):
            legal = st.legal_actions()
            st.apply_action(legal[int(rng.integers(len(legal)))])
        out.append(st)
    return out


def root_edges(root, n, en, ew):
    """A harness dump's root edges as [n*n] visits / sums by action."""
    legal = root.legal_actions()
    v, s = np.zeros(n * n, dtype=np.int32), np.zeros(n * n, dtype=np.float64)
    v[legal], s[legal] = en[0, :len(legal)], ew[0, :len(legal)]
    return v, s


# --------------------------------------------------------------------- host harnesses vs specifications ---
# line_roots seeds whose lines end in wins as well as draws: n = 8 -> 5, n = 12 -> 1, n = 24 -> 0
ROOT_SEED = {8: 5, 12: 1, 24: 0}


@pytest.mark.parametrize("n,sims,min_depth", [(8, 120, 33), (12, 200, 65)])
def test_puct_line_harness_matches_spec(ph, oracle_mod, n, sims, min_depth):  # noqa: F811
    checked, deepest = 0, 0
    for i, root in enumerate(line_roots(oracle_mod.OracleGame(n), 4, ROOT_SEED[n])):
        ev = Evaluator(n, "puct")
        ref = puct_spec.Search(root, tp.SEED, 7 + i, 1, 50.0)
        drive(ref, sims, ev)
        depth, terminals, _ = reach(ref)
        assert depth >= 33 and terminals >= 1, i
        deepest = max(deepest, depth)
        got = tp.harness_search(ph, root, n, tp.SEED, 7 + i, 1, 50.0, sims, ev.value, ev.prior)
        tp.assert_harness_matches(got, ref, n, (n, i))
        checked += check_puct_line_root(root, n, sims, *root_edges(root, n, got[5], got[6]))
    assert checked >= 1 and deepest >= min_depth


def _vh_line(vh, kind, root, n, T, c, vl, sims, K, ev, R=1):  # noqa: F811
    """The virtual-loss harness and its specification in lock step on the evaluator (K = 1: the plain UCT / PUCT
    search); every leaf at every step, then every node."""
    rec = np.ascontiguousarray(root.export_record())
    ref = tv.make(kind, root, tv.SEED, T, R, c, vl)
    h = vh.vh_create(P(rec), n, tv.SEED, T, R, c, sims, int(kind == "puct"), K, vl)
    S, M = sims + 1, n * (n - 2)
    leaves = np.zeros((K, rec.size), dtype=np.uint32)
    slots, status = np.zeros(K, dtype=np.int32), np.zeros(K, dtype=np.int32)
    a = dict(parent=np.zeros(S, np.int32), action=np.zeros(S, np.int32), nn=np.zeros(S, np.uint32),
             nv=np.zeros(S, np.uint32), legal=np.zeros(S, np.int32), en=np.zeros((S, M), np.uint32),
             ew=np.zeros((S, M), np.float64), ev=np.zeros((S, M), np.uint32), ep=np.zeros((S, M), np.float32),
             best=np.zeros(1, np.int32))
    try:
        for step in range(sims // K):
            count = vh.vh_select_step(h, P(leaves), P(slots), P(status))
            got = ref.select_step(K)
            assert [(int(x), bool(y)) for x, y in zip(slots, status)] == got, step
            assert count == len(ref.nodes), step
            vals = np.zeros((K, 2), dtype=np.float32)
            pri = np.full((K, n * n), 1.0 / (n * n), dtype=np.float32)
            sv, sp = [], []
            for j, (leaf, terminal) in enumerate(got):
                st = ref.nodes[leaf].state
                assert np.array_equal(leaves[j], st.export_record()), (step, j)
                if terminal:
                    sv.append(None)
                    sp.append(None)
                    continue
                v, p = ev(st)
                vals[j] = v
                if p is not None:
                    pri[j] = p
                sv.append(v)
                sp.append(p)
            vh.vh_backup_step(h, P(vals), P(pri))
            ref.backup_step(sv, sp) if kind == "puct" else ref.backup_step(sv)
        nodes = vh.vh_dump(h, P(a["parent"]), P(a["action"]), P(a["nn"]), P(a["nv"]), P(a["legal"]), P(a["en"]),
                           P(a["ew"]), P(a["ev"]), P(a["ep"]), P(a["best"]))
    finally:
        vh.vh_destroy(h)
    d = tv.dump(kind, ref)
    assert nodes == len(d)
    assert not a["nv"][:nodes].any() and not a["ev"][:nodes].any()
    for s_, row in enumerate(d):
        par, act, nn, L, e_n, e_w = row[:6]
        assert (a["parent"][s_], a["action"][s_], a["nn"][s_], a["legal"][s_]) == (par, act, nn, L), s_
        if L > 0:
            assert a["en"][s_, :L].tolist() == list(e_n), s_
            assert a["ew"][s_, :L].tobytes() == np.asarray(e_w, dtype=np.float64).tobytes(), s_
            if kind == "puct":
                assert a["ep"][s_, :L].tobytes() == np.asarray(row[6], dtype=np.float32).tobytes(), s_
    assert int(a["best"][0]) == ref.root_stats(n)[2]
    return ref


@pytest.mark.parametrize("n,sims", [(7, 900), (8, 1200)])
def test_uct_line_harness_matches_spec(vh, oracle_mod, n, sims):  # noqa: F811
    """uct_c = 0 and values (1, 1): a node's children are swept once, then the descent takes the lowest edge.  At
    n = 7 the line runs into won terminals near depth 20 and stays there; n = 8 goes past depth 33."""
    root = oracle_mod.OracleGame(n).new_initial_state()
    ref = _vh_line(vh, "uct", root, n, 3, 0.0, 1.0, sims, 1, Evaluator(n, "uct"))
    assert_uct_line_reach([ref], n)


@pytest.mark.parametrize("K,vl", [(4, 50.0), (33, 0.0), (64, 1.0)])
def test_virtual_loss_line_harness_matches_spec(vh, oracle_mod, K, vl):  # noqa: F811
    n, steps = 8, 36
    root = oracle_mod.OracleGame(n).new_initial_state()
    ref = _vh_line(vh, "puct", root, n, 11 + K, 50.0, vl, steps * K, K, Evaluator(n, "puct"))
    assert reach(ref)[0] >= 33


def test_solver_puct_line_harness_matches_spec(sh, oracle_mod):  # noqa: F811
    """The line runs into a won terminal deeper than 32: the proof walk starts there."""
    n, sims = 8, 120
    root = oracle_mod.OracleGame(n).new_initial_state()
    ev = Evaluator(n, "puct")
    ref = solver_spec.make("puct", root, ts.SEED, 5, 1, 50.0)
    statuses = drive(ref, sims, ev)
    depth, terminals, _ = reach(ref)
    assert depth > 32 and terminals >= 1 and 1 in statuses
    got = ts.harness_search(sh, "puct", root, n, ts.SEED, 5, 1, 50.0, sims, ev.value, ev.prior)
    ts.assert_harness_matches(got, ref, statuses, n, "line")


@pytest.mark.parametrize("n,sims,mc,min_depth", [(8, 120, 1, 33), (12, 200, 1, 65), (8, 160, 16, 33)])
def test_gumbel_line_harness_matches_spec(gh, oracle_mod, n, sims, mc, min_depth):  # noqa: F811
    """max_considered = 1, zero root noise and +20 on the line's move; mc = 16 spreads the root over 16 moves (logits
    in [0, 1.5] on the others) whose subtrees still follow the line."""
    root = oracle_mod.OracleGame(n).new_initial_state()
    ev = Evaluator(n, "gumbel" if mc == 1 else "gumbel-spread")
    ref = gumbel_spec.Search(root, tg.SEED, 9, 1, sims, mc)
    drive(ref, sims, ev)
    assert reach(ref)[0] >= min_depth
    if mc > 1:
        assert np.count_nonzero(ref.root_stats(n)[0]) >= 8
    got = tg.harness_search(gh, root, n, 9, 1, sims, mc, None, ev.value, ev.prior)
    tg.assert_harness_matches(got, ref, n, (n, mc))


# ---------------------------------------------------------------------------------------------- GPU ---
def _batch(roots, n, seed, extra=0):
    from twixt_for_open_spiel_b200 import TwixTBatch
    b = TwixTBatch(n, len(roots) + extra, 0, seed)
    b.import_state(np.stack([r.export_record() for r in roots]), 0)
    return b


def _lockstep(m, b, refs, n, ev, sims, on_step=None):
    """K = 1: the device search and the specifications in lock step on the evaluator, with every leaf record and
    status compared at every step.  Rows of terminal leaves and finished trees get zero values and uniform priors,
    which the search ignores.  on_step(k, leaves, statuses) sees each step."""
    trees, uct = len(refs), m.selection == "uct"
    for k in range(sims):
        status = m.select(trees)
        leaves = b.export_state(trees, trees)
        values = np.zeros((trees, 2), dtype=np.float32)
        rows = np.full((trees, n * n), 1.0 / (n * n), dtype=np.float32)
        if m.selection == "gumbel":
            rows[:] = 0.0
        for t, ref in enumerate(refs):
            leaf, st = ref.select()
            assert status[t] == int(st), (n, k, t)
            if st != solver_spec.LEAF_SOLVED:
                assert np.array_equal(leaves[t], ref.nodes[leaf].state.export_record()), (n, k, t)
            if st:
                ref.backup(*((None,) if uct else (None, None)))
                continue
            v, p = ev(ref.nodes[leaf].state)
            values[t] = v
            if p is not None:
                rows[t] = p
            ref.backup(*((v,) if uct else (v, p)))
        if on_step is not None:
            on_step(k, leaves, status)
        m.backup(values, None if uct else rows)


def _continue_run(m, b, refs, extra, counter):
    """`run(extra)` with the built-in rollouts on the device and on the (counted) specifications."""
    b.stats_reset()
    m.run(extra)
    for ref in refs:
        counter.wrap(ref)
        if isinstance(ref, (vl_spec.PuctSearch, vl_spec.UctSearch)):
            ref.run_steps(extra, m.leaves_per_step)
        else:
            ref.run(extra)
    st = b.stats()
    assert (st["plies"], st["games"]) == (counter.plies, counter.games)


@pytest.mark.gpu
@pytest.mark.parametrize("n,trees,sims,extra,R,min_depth", [
    (8, 4, 120, 8, 33, 33), (12, 4, 200, 8, 64, 65),
    (12, 4, 140, 0, 1, 139),  # max_simulations 140 < max_game_length 141: P = 141, the line reaches depth 139
    (24, 2, 600, 4, 33, 571)])  # a full game (a draw at ply 571) and a win at ply 394
def test_device_puct_line_matches_spec(oracle_mod, n, trees, sims, extra, R, min_depth):
    """The PUCT line stepwise (uct_c = 50), then `run(extra)` with R rollouts per leaf from its deep leaves."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    roots = line_roots(oracle_mod.OracleGame(n), trees, ROOT_SEED[n])
    b = _batch(roots, n, tp.SEED, extra=trees)
    b.set_stream_base(40)
    m = BatchedMCTS(b, trees, sims + extra, R, 50.0, selection="puct")
    m.begin(0, trees)
    refs = [puct_spec.Search(r, tp.SEED, 40 + t, R, 50.0) for t, r in enumerate(roots)]
    ev = Evaluator(n, "puct")
    lines = [oracle_line(r, sims) for r in roots]
    first_terminal = [None] * trees

    def independent(k, leaves, status):  # simulation k's leaf is the line's state after min(k, end) moves
        for t, line in enumerate(lines):
            if first_terminal[t] is None:
                assert np.array_equal(leaves[t], line[min(k, len(line) - 1)].export_record()), (k, t)
                if status[t]:
                    first_terminal[t] = k
    _lockstep(m, b, refs, n, ev, sims, independent)
    visits, sums, best = m.root_stats()
    tp._assert_stats_equal((visits, sums, best), refs, n, "line")
    checked = sum(check_puct_line_root(r, n, sims, visits[t], sums[t]) for t, r in enumerate(roots))
    reached = [reach(ref) for ref in refs]
    assert max(d for d, _, _ in reached) >= min_depth and min(d for d, _, _ in reached) >= 33, reached
    if n == 12 and sims == 140:
        assert max(d for d, _, _ in reached) == m.max_simulations - 1 < 141
    else:
        assert checked >= 1 and all(t >= 1 for _, t, _ in reached), reached
    if extra:
        _continue_run(m, b, refs, extra, tr._Counted())
        tp._assert_stats_equal(m.root_stats(), refs, n, "run")


@pytest.mark.gpu
@pytest.mark.parametrize("n,trees,sims,solve", [(7, 4, 900, True), (8, 3, 1200, False)])
def test_device_uct_line_matches_spec(oracle_mod, n, trees, sims, solve):
    """The UCT line (uct_c = 0, values (1, 1)) stepwise, then `run(16)` with 64 rollouts per leaf.  At n = 7 it
    runs into won terminals, so the solver search is the one tested there."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    roots = line_roots(oracle_mod.OracleGame(n), trees, n)
    b = _batch(roots, n, tr.SEED, extra=trees)
    m = BatchedMCTS(b, trees, sims + 16, 64, 0.0, selection="uct", solve=solve)
    m.begin(0, trees)
    refs = [tr.make("uct", solve, r, t, 64, 0.0) for t, r in enumerate(roots)]
    _lockstep(m, b, refs, n, Evaluator(n, "uct"), sims)
    tr._assert_same(m, refs, n, "line")
    assert_uct_line_reach(refs, n)
    _continue_run(m, b, refs, 16, tr._Counted())
    tr._assert_same(m, refs, n, "run")


@pytest.mark.gpu
@pytest.mark.parametrize("n,trees,sims", [(8, 4, 120), (12, 2, 200)])
def test_device_solver_puct_line_matches_spec(oracle_mod, n, trees, sims):
    """MCTS-Solver on the PUCT line: proof walks that start at terminals deeper than 32, then `run(8)` with 33
    rollouts per leaf."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    roots = line_roots(oracle_mod.OracleGame(n), trees, ROOT_SEED[n])
    b = _batch(roots, n, ts.SEED, extra=trees)
    m = BatchedMCTS(b, trees, sims + 8, 33, 50.0, selection="puct", solve=True)
    m.begin(0, trees)
    refs = [solver_spec.make("puct", r, ts.SEED, t, 33, 50.0) for t, r in enumerate(roots)]
    _lockstep(m, b, refs, n, Evaluator(n, "puct"), sims)
    ts._assert_stats_equal(m, refs, n, "line")
    for ref in refs:
        depth, terminals, _ = reach(ref)
        assert terminals >= 1 and depth > 32
        deepest_terminal = max(d for d, nd in zip(_depths(ref), ref.nodes) if nd.state.is_terminal())
        assert deepest_terminal > 32
    _continue_run(m, b, refs, 8, tr._Counted())
    ts._assert_stats_equal(m, refs, n, "run")


def _depths(ref):
    depth = [0] * len(ref.nodes)
    for i, nd in enumerate(ref.nodes[1:], 1):
        depth[i] = depth[nd.parent_slot if _is_puct_family(ref) else nd.parent] + 1
    return depth


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uct", "puct"])
@pytest.mark.parametrize("R", [33, 64])
def test_device_solver_trees_finish_with_wide_rollouts(oracle_mod, kind, R):
    """Solver trees that finish during `run` while R > 32: the finished tree's rollout slots (all R of them) are
    counted as neither plies nor games."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 24, 40
    roots = solver_spec.near_end_roots(oracle_mod.OracleGame(n), n, 31 + R, trees, back=(1, 2, 3))
    b = _batch(roots, n, ts.SEED)
    m = BatchedMCTS(b, trees, sims, R, 2.0, selection=kind, solve=True)
    m.begin(0, trees)
    refs = [solver_spec.make(kind, r, ts.SEED, t, R, 2.0) for t, r in enumerate(roots)]
    _continue_run(m, b, refs, sims, tr._Counted())
    ts._assert_stats_equal(m, refs, n, (kind, R))
    assert sum(r.finished for r in refs) >= trees // 4


@pytest.mark.gpu
@pytest.mark.parametrize("K", [4, 33, 64])
@pytest.mark.parametrize("vl", [0.0, 1.0, 50.0])
def test_device_virtual_loss_line_matches_spec(oracle_mod, K, vl):
    """K descents per step on the PUCT line: with vl = 0 all of them follow the line to the same deep leaf, with 50
    they branch off at many depths.  Then `run(2K)` with 33 rollouts per leaf (K * R > 32)."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, steps, R = 8, 2, 36, 33
    roots = line_roots(oracle_mod.OracleGame(n), trees + 1, ROOT_SEED[n])[1:]
    b = _batch(roots, n, tv.SEED, extra=trees * K)
    m = BatchedMCTS(b, trees, (steps + 2) * K, R, 50.0, selection="puct", leaves_per_step=K, virtual_loss=vl)
    m.begin(0, trees)
    refs = [tv.make("puct", r, tv.SEED, t, R, 50.0, vl) for t, r in enumerate(roots)]
    ev = Evaluator(n, "puct")
    rows = trees * K
    for step in range(steps):
        status = m.select(trees)
        leaves = b.export_state(trees, rows)
        values = np.zeros((rows, 2), dtype=np.float32)
        priors = np.full((rows, n * n), 1.0 / (n * n), dtype=np.float32)
        for t, ref in enumerate(refs):
            got = ref.select_step(K)
            sv, sp = [], []
            for j, (leaf, terminal) in enumerate(got):
                st = ref.nodes[leaf].state
                assert status[t * K + j] == int(terminal), (step, t, j)
                assert np.array_equal(leaves[t * K + j], st.export_record()), (step, t, j)
                v, p = (None, None) if terminal else ev(st)
                if not terminal:
                    values[t * K + j], priors[t * K + j] = v, p
                sv.append(v)
                sp.append(p)
            ref.backup_step(sv, sp)
        m.backup(values, priors)
    tv._assert_stats_equal(m.root_stats(), refs, n, (K, vl))
    for ref in refs:
        depth, _, nodes = reach(ref)
        assert depth >= 33
        assert nodes == depth + 1 if vl == 0.0 else True
    if vl == 50.0:
        assert max(reach(ref)[2] for ref in refs) > 2 * steps
    _continue_run(m, b, refs, 2 * K, tr._Counted())
    tv._assert_stats_equal(m.root_stats(), refs, n, (K, vl, "run"))


@pytest.mark.gpu
@pytest.mark.parametrize("keep", ["S", 40, 33, 2])
def test_device_advance_along_the_line_matches_spec(oracle_mod, keep):
    """Tree reuse on the PUCT line: 60 simulations, advance along the line's first move keeping `keep` nodes, then
    simulations up to the arena's capacity, all stepwise."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, cap, sims = 8, 3, 80, 60
    S = cap + 1
    keep = S if keep == "S" else keep
    roots = line_roots(oracle_mod.OracleGame(n), trees + 1, ROOT_SEED[n])[1:]
    b = _batch(roots, n, tr.SEED, extra=trees)
    m = BatchedMCTS(b, trees, cap, 1, 50.0, selection="puct")
    m.begin(0, trees)
    refs = [tr.make("puct", False, r, t, 1, 50.0) for t, r in enumerate(roots)]
    ev = Evaluator(n, "puct")
    _lockstep(m, b, refs, n, ev, sims)
    assert all(reach(ref)[0] >= 33 for ref in refs)
    actions = np.asarray([line_action(r) for r in roots], dtype=np.int32)
    status = m.advance(actions, keep)
    assert status.tolist() == [reuse_spec.advance(ref, int(a), keep) for ref, a in zip(refs, actions)]
    tr._assert_same(m, refs, n, "advanced")
    kept = [len(ref.nodes) for ref in refs]
    assert max(kept) == min(keep, sims - 1)
    # the host's node bound after the advance is min(keep, 1 + sims)
    _lockstep(m, b, refs, n, ev, S - min(keep, sims + 1))
    tr._assert_same(m, refs, n, "searched again")
    assert all(reach(ref)[0] >= 33 for ref in refs)


@pytest.mark.gpu
def test_device_tree_fills_the_arena_and_the_path(oracle_mod):
    """One tree driven to S = max_simulations + 1 nodes and a leaf at depth max_simulations: the line for
    max_simulations simulations (max_simulations nodes), an advance that keeps the root and all those nodes (which
    brings the host's node bound down to them), and one more simulation."""
    from twixt_for_open_spiel_b200.mcts import ROOT_KEPT, BatchedMCTS
    n, cap = 12, 100
    root = line_roots(oracle_mod.OracleGame(n), 2, ROOT_SEED[n])[1]
    assert len(oracle_line(root, cap + 1)) == cap + 2  # the line is longer than the arena
    b = _batch([root], n, tr.SEED, extra=1)
    m = BatchedMCTS(b, 1, cap, 1, 50.0, selection="puct")
    m.begin(0, 1)
    ref = tr.make("puct", False, root, 0, 1, 50.0)
    ev = Evaluator(n, "puct")
    _lockstep(m, b, [ref], n, ev, cap)
    assert reach(ref) == (cap - 1, 0, cap)
    assert m.advance(np.asarray([-1], dtype=np.int32), cap).tolist() == [ROOT_KEPT]
    assert reuse_spec.advance(ref, -1, cap) == ROOT_KEPT
    _lockstep(m, b, [ref], n, ev, 1)
    assert reach(ref) == (cap, 0, cap + 1)
    tr._assert_same(m, [ref], n, "full")
    with pytest.raises(ValueError):
        m.run(1)


def improved_policy_f64(logits, visits, sums, raw_value, c_visit=50.0, c_scale=0.1):
    """softmax(logits + sigma(completed Q)) in float64 numpy (mctx qtransform_completed_by_mix_value)."""
    logits = np.asarray(logits, dtype=np.float64)
    visits = np.asarray(visits, dtype=np.float64)
    pi = np.exp(logits - logits.max())
    pi /= pi.sum()
    seen = visits > 0
    q = np.where(seen, np.asarray(sums) / np.maximum(visits, 1), 0.0)
    sum_n = visits.sum()
    weighted = (pi[seen] * q[seen]).sum() / pi[seen].sum() if sum_n > 0 else 0.0
    v_mix = (raw_value + sum_n * weighted) / (sum_n + 1.0)
    q = np.where(seen, q, v_mix)
    q = (q - q.min()) / max(q.max() - q.min(), 1e-8)
    x = logits + (c_visit + visits.max()) * c_scale * q
    e = np.exp(x - x.max())
    return e / e.sum()


@pytest.mark.gpu
@pytest.mark.parametrize("n,trees,sims,mc,extra,R,min_depth", [
    (8, 4, 120, 1, 8, 33, 33), (12, 2, 200, 1, 8, 64, 65), (24, 1, 60, 1, 0, 1, 33), (8, 4, 160, 16, 8, 33, 33)])
def test_device_gumbel_line_matches_spec(oracle_mod, n, trees, sims, mc, extra, R, min_depth):
    """The Gumbel line: zero root noise, +20 on the line's move (mc = 16: the other logits in [0, 1.5], so Sequential
    Halving spreads the root while each subtree follows the line), then `run(extra)` with R rollouts per leaf."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    roots = line_roots(oracle_mod.OracleGame(n), trees, ROOT_SEED[n])
    b = _batch(roots, n, tg.SEED, extra=trees)
    m = BatchedMCTS(b, trees, sims + extra, R, selection="gumbel", max_considered=mc)
    m.begin(0, trees)
    refs = [gumbel_spec.Search(r, tg.SEED, t, R, sims + extra, mc) for t, r in enumerate(roots)]
    ev = Evaluator(n, "gumbel" if mc == 1 else "gumbel-spread")
    _lockstep(m, b, refs, n, ev, sims)
    tg._assert_matches(m, refs, n, "line")
    reached = [reach(ref) for ref in refs]
    assert max(d for d, _, _ in reached) >= min_depth and min(d for d, _, _ in reached) >= 33, reached
    visits, sums, _ = m.root_stats()
    _, policy = m.gumbel_stats()
    for t, root in enumerate(roots):
        legal = root.legal_actions()
        v, logits = ev(root)
        want = improved_policy_f64(logits[legal], visits[t, legal], sums[t, legal],
                                   float(v[int(root.export_record()[0]) & 1]))
        got = policy[t, legal].astype(np.float64)
        assert np.allclose(got, want, rtol=2 ** -22, atol=1e-44), t
        assert not np.any(np.delete(policy[t], legal))
        if mc == 1:
            assert np.count_nonzero(visits[t]) == 1 and visits[t, line_action(root)] == sims - 1
        else:
            assert np.count_nonzero(visits[t]) >= 8
    if extra:
        _continue_run(m, b, refs, extra, tr._Counted())
        tg._assert_matches(m, refs, n, "run")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uct", "puct", "gumbel"])
@pytest.mark.parametrize("R", [33, 64])
def test_device_run_with_wide_rollouts_matches_spec(oracle_mod, kind, R):
    """`run` with R > 32 rollouts per leaf (the rollout-id loops take a second lane pass) from roots of every kind,
    twixt_stats included."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 12, 40
    roots = mcts_spec.root_positions(oracle_mod.OracleGame(n), n, R + len(kind), trees)
    b = _batch(roots, n, tr.SEED)
    b.set_stream_base(900)
    m = BatchedMCTS(b, trees, sims, R, 1.25, selection=kind)
    m.begin(0, trees)
    if kind == "gumbel":
        refs = [gumbel_spec.Search(r, tr.SEED, 900 + t, R, sims, 16) for t, r in enumerate(roots)]
    else:
        refs = [tr.make(kind, False, r, 900 + t, R, 1.25) for t, r in enumerate(roots)]
    _continue_run(m, b, refs, sims, tr._Counted())
    if kind == "gumbel":
        tg._assert_matches(m, refs, n, R)
    else:
        tr._assert_same(m, refs, n, (kind, R))
