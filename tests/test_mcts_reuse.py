"""Tree reuse across moves (twixt_mcts_advance, twixt_mcts_set_root_priors, BatchedMCTS.advance,
MCTSBot(reuse_tree=True)) against its executable specification tests/reuse_spec.py.  CPU: the specification's own
properties.  GPU: the device search bit for bit against the specification for every kind, after the advance, after
more simulations and in the stepwise form, plus chains over whole games, pointers, errors, budgets, launch counts,
the bot, the self-play example and a search at scale."""
import os
import random
import sys

import numpy as np
import pytest

import mcts_spec
import puct_spec
import reuse_spec
import solver_spec

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SEED = 0x72657573
KINDS = [("uct", False), ("puct", False), ("uct", True), ("puct", True)]
KIND_IDS = ["uct", "puct", "uct-solve", "puct-solve"]


def make(kind, solve, root, T, R=1, c=2.0, K=1, vl=1.0):
    return reuse_spec.make(kind, root, SEED, T, R, c, solve, K, vl)


def spec_run(ref, sims, K, value_fn=None, prior_fn=None):
    if K > 1:
        return ref.run_steps(sims, K, value_fn, *(() if prior_fn is None else (prior_fn,)))
    if isinstance(ref, puct_spec.Search):
        return ref.run(sims, value_fn, prior_fn)
    return ref.run(sims, value_fn)


def root_state(ref):
    return ref.nodes[0].state


def ply(state):
    return int(state.export_record()[0])


def ending_move(state):
    for a in state.legal_actions():
        ch = state.clone()
        ch.apply_action(a)
        if ch.is_terminal():
            return a
    return None


def choose(ref, n, t, rng):
    """Tree t's action by category t % 6: the best move, a visited non-best move, an unvisited legal move, the
    swap at ply 1, -1, a move that ends the game (each falls back to the best move, or -1, where it does not
    exist)."""
    st = root_state(ref)
    if st.is_terminal():
        return -1
    visits, _, best = ref.root_stats(n)
    legal = st.legal_actions()
    fallback = best if best >= 0 else legal[0]
    cat = t % 6
    if cat == 1:
        other = [a for a in legal if visits[a] > 0 and a != best]
        return rng.choice(other) if other else fallback
    if cat == 2:
        free = [a for a in legal if visits[a] == 0]
        return rng.choice(free) if free else fallback
    if cat == 3:
        first = int(st.export_record()[2])
        return first if ply(st) == 1 and first in legal else fallback
    if cat == 4:
        return -1
    if cat == 5:
        a = ending_move(st)
        return fallback if a is None else a
    return fallback


# ------------------------------------------------------------------------------- the specification itself ---
def _searched(kind, solve, K, n, count, sims, seed):
    g = __import__("oracle").pyoracle.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, seed, count)
    return [spec_run(make(kind, solve, r, 50 + t, 1, 1.5, K), sims, K, mcts_spec.stand_in_value,
                     (lambda rec: puct_spec.stand_in_priors(rec, n)) if kind == "puct" else None)
            for t, r in enumerate(roots)]


def _subtree_stats(ref, start):
    """[(N(s), sorted edge (action, N, W) list)] of the subtree of slot `start`, in slot order."""
    out = []
    if isinstance(ref, puct_spec.Search):
        want = {start}
        for nd in ref.nodes[start:]:
            if nd.slot in want:
                out.append((nd.explore_count, [(c.action, c.explore_count, c.total_reward) for c in nd.edges()]))
                want.update(c.slot for c in nd.children if c.slot is not None)
    else:
        want = {start}
        for i in range(start, len(ref.nodes)):
            if i in want:
                nd = ref.nodes[i]
                out.append((nd.n, list(zip(nd.actions or [], nd.edge_n, nd.edge_w))))
                want.update(c for c in nd.children if c >= 0)
    return out


def _child_slot(ref, action):
    if isinstance(ref, puct_spec.Search):
        c = next((c for c in ref.nodes[0].children if c.action == action), None)
        return None if c is None else c.slot
    nd = ref.nodes[0]
    if nd.actions is None:
        return None
    c = nd.children[nd.actions.index(action)]
    return None if c < 0 else c


@pytest.mark.parametrize("kind,solve", KINDS, ids=KIND_IDS)
@pytest.mark.parametrize("K", [1, 3])
def test_spec_full_keep_preserves_the_subtree(oracle_mod, kind, solve, K):
    if solve and K > 1:
        pytest.skip("the solver runs one leaf per step")
    n, sims = 8, 48
    rng = random.Random(1)
    for t, ref in enumerate(_searched(kind, solve, K, n, 12, sims, 7)):
        a = choose(ref, n, t, rng)
        start = 0 if a == -1 else _child_slot(ref, a)
        before = _subtree_stats(ref, start) if start is not None else None
        status = reuse_spec.advance(ref, a, sims + 1)
        reuse_spec.check_tree(ref)
        if before is not None:
            assert _subtree_stats(ref, 0) == before
            assert reuse_spec.node_count(ref) == len(before)
            assert status == (reuse_spec.ROOT_KEPT if before[0][0] > 0 else reuse_spec.ROOT_FRESH)
        elif a != -1:
            assert status == reuse_spec.ROOT_FRESH and reuse_spec.node_count(ref) == 1


@pytest.mark.parametrize("kind,solve", KINDS, ids=KIND_IDS)
@pytest.mark.parametrize("keep", [1, 2, 3, 7])
def test_spec_cap_gives_a_rooted_tree_with_unvisited_dropped_edges(oracle_mod, kind, solve, keep):
    n, sims = 8, 64
    rng = random.Random(keep)
    for t, ref in enumerate(_searched(kind, solve, 1, n, 12, sims, 9)):
        a = choose(ref, n, t, rng)
        start = 0 if a == -1 else _child_slot(ref, a)
        before = _subtree_stats(ref, start) if start is not None else None
        reuse_spec.advance(ref, a, keep)
        reuse_spec.check_tree(ref)
        assert reuse_spec.node_count(ref) <= keep
        if before is None:
            continue
        assert reuse_spec.node_count(ref) == min(keep, len(before))
        # every kept node keeps N(s); an edge keeps (N, W) exactly when it still has its child
        after = _subtree_stats(ref, 0)
        for (nb, eb), (na, ea) in zip(before, after):
            assert nb == na
        if isinstance(ref, puct_spec.Search):
            for nd in ref.nodes:
                for c in nd.children:
                    if c.slot is None:
                        assert (c.explore_count, c.total_reward, c.children) == (0, 0.0, [])
        else:
            for nd in ref.nodes:
                for i, c in enumerate(nd.children):
                    if c < 0:
                        assert (nd.edge_n[i], nd.edge_w[i]) == (0, 0.0)


def test_spec_hand_traced_advance(oracle_mod):
    """n = 5, UCT.  Slots 0..5: the root with children 1 (action a) and 2 (action b); 1 has children 3 and 5, 2 has
    child 4.  Advancing along a keeps 1, 3, 5 as 0, 1, 2; with keep = 2 slot 5 is dropped and its edge in node 1
    is unvisited again."""
    g = oracle_mod.OracleGame(5)
    for keep, expect in ((6, [1, 3, 5]), (2, [1, 3])):
        s = mcts_spec.Search(g.new_initial_state(), SEED, 0)
        root = s.nodes[0]
        root.n = 5
        root.actions = root.state.legal_actions()
        a, b = root.actions[0], root.actions[1]
        L = len(root.actions)
        root.edge_n, root.edge_w, root.children = [0] * L, [0.0] * L, [-1] * L

        def add(parent, e):
            p = s.nodes[parent]
            st = p.state.clone()
            st.apply_action(p.actions[e])
            s.nodes.append(mcts_spec.Node(st, parent, p.actions[e]))
            p.children[e] = len(s.nodes) - 1
            return len(s.nodes) - 1

        def expand(i, n_visits):
            nd = s.nodes[i]
            nd.n = n_visits
            nd.actions = nd.state.legal_actions()
            m = len(nd.actions)
            nd.edge_n, nd.edge_w, nd.children = [0] * m, [0.0] * m, [-1] * m

        add(0, 0)
        add(0, 1)
        root.edge_n[0], root.edge_w[0], root.edge_n[1], root.edge_w[1] = 3, 0.5, 1, -1.0
        expand(1, 3)
        add(1, 2)
        s.nodes[1].edge_n[2], s.nodes[1].edge_w[2] = 1, 0.25
        s.nodes[2].n = 1
        expand(2, 1)
        add(2, 0)
        s.nodes[3].n = 1
        add(1, 4)
        s.nodes[1].edge_n[4], s.nodes[1].edge_w[4] = 1, -0.75
        s.nodes[4].n, s.nodes[5].n = 0, 1
        s.k = 5
        old = list(s.nodes)
        assert reuse_spec.advance(s, a, keep) == reuse_spec.ROOT_KEPT
        assert s.nodes == [old[i] for i in expect] and s.k == 5
        r = s.nodes[0]
        assert (r.parent, r.action, r.n) == (-1, -1, 3)
        assert r.children[2] == 1 and r.edge_n[2] == 1 and r.edge_w[2] == 0.25
        if keep == 6:
            assert r.children[4] == 2 and (r.edge_n[4], r.edge_w[4]) == (1, -0.75) and s.nodes[2].parent == 0
        else:
            assert r.children[4] == -1 and (r.edge_n[4], r.edge_w[4]) == (0, 0.0)
    s = mcts_spec.Search(g.new_initial_state(), SEED, 0)
    assert reuse_spec.advance(s, b, 5) == reuse_spec.ROOT_FRESH  # the root is not expanded: a fresh root
    moved = g.new_initial_state()
    moved.apply_action(b)
    assert len(s.nodes) == 1 and np.array_equal(s.nodes[0].state.export_record(), moved.export_record())
    assert reuse_spec.advance(s, 10 ** 6, 5) == reuse_spec.ROOT_ILLEGAL


@pytest.mark.parametrize("kind", ["uct", "puct"])
def test_spec_solver_root_code_matches_negamax(oracle_mod, kind):
    """Advancing into proven children at n = 5 gives the root the child's exact value."""
    n = 5
    g = oracle_mod.OracleGame(n)
    memo = {}
    roots = solver_spec.near_end_roots(g, n, 11, 40, back=(2, 3, 4))
    seen = {1: 0, 2: 0, 3: 0}
    for t, root in enumerate(roots):
        if root.is_terminal():
            continue
        ref = make(kind, True, root, t)
        ref.run(120)
        codes = ref.edge_codes(0) if kind == "uct" else ref.edge_codes(ref.nodes[0])
        acts = root.legal_actions()
        for e, c in enumerate(codes):
            if c == 0:
                continue
            r2 = make(kind, True, root, t)
            r2.run(120)
            reuse_spec.advance(r2, acts[e], 200)
            child = root.clone()
            child.apply_action(acts[e])
            assert r2.root_code() == 2 + solver_spec.negamax(child, memo)
            assert r2.root_code() == 4 - c
            assert r2.finished
            seen[c] += 1
            break
    assert seen[1] + seen[2] + seen[3] > 0 and seen[3] + seen[1] > 0, seen


@pytest.mark.parametrize("kind,solve", KINDS, ids=KIND_IDS)
def test_spec_advance_then_search_is_deterministic(oracle_mod, kind, solve):
    n = 8
    out = []
    for _ in range(2):
        refs = _searched(kind, solve, 1, n, 6, 32, 3)
        rng = random.Random(5)
        for t, ref in enumerate(refs):
            reuse_spec.advance(ref, choose(ref, n, t, rng), 20)
            spec_run(ref, 24, 1)
            reuse_spec.check_tree(ref)
        out.append([ref.root_stats(n) for ref in refs])
    for x, y in zip(*out):
        assert all(np.array_equal(a, b) for a, b in zip(x[:2], y[:2])) and x[2] == y[2]


# ---------------------------------------------------------------------------------------------- GPU ---
def _batch_with_roots(roots, n, extra=0, seed=SEED):
    from twixt_for_open_spiel_b200 import TwixTBatch
    b = TwixTBatch(n, len(roots) + extra, 0, seed)
    b.import_state(np.stack([r.export_record() for r in roots]), 0)
    return b


def _assert_same(m, refs, n, tag):
    visits, sums, best = m.root_stats()
    for t, ref in enumerate(refs):
        v, w, bst = ref.root_stats(n)
        assert np.array_equal(visits[t], v), (tag, t)
        assert sums[t].tobytes() == w.tobytes(), (tag, t)
        assert best[t] == bst, (tag, t)
    if m.solve:
        got = m.solver_stats()
        for t, ref in enumerate(refs):
            want = ref.solver_stats(n)
            assert got[0][t] == want[0], (tag, t)
            assert got[1][t].tobytes() == want[1].tobytes(), (tag, t)
            assert np.array_equal(got[2][t], want[2]), (tag, t)
            assert got[3][t] == want[3], (tag, t)


class _Counted:
    """Counts the plies and games of a specification's rollouts (what twixt_stats must add)."""

    def __init__(self):
        self.plies = 0
        self.games = 0

    def wrap(self, s):
        def count(leaf, k):
            for r in range(s.R):
                st = s.nodes[leaf].state.clone()
                self.plies += len(st.playout_philox(s.seed, mcts_spec.rollout_stream(s.T, k, s.R, r)))
                self.games += 1
        if hasattr(s, "rollout_value_at"):
            orig_at = s.rollout_value_at

            def rollout_value_at(leaf, k):
                count(leaf, k)
                return orig_at(leaf, k)
            s.rollout_value_at = rollout_value_at
        else:
            orig = s.rollout_value

            def rollout_value(leaf):
                count(leaf, s.k)
                return orig(leaf)
            s.rollout_value = rollout_value
        return s


CASES = [(kind, solve, K) for kind, solve in KINDS for K in (1, 4) if not (solve and K > 1)]
CASE_IDS = ["%s-K%d" % (KIND_IDS[KINDS.index((k, s))], K) for k, s, K in CASES]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,solve,K", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("n,trees,sims", [(5, 18, 48), (8, 18, 32), (12, 12, 24), (24, 6, 16)])
@pytest.mark.parametrize("cap", ["S", 3, 1])
def test_device_advance_and_run_match_spec(oracle_mod, kind, solve, K, n, trees, sims, cap):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 5 * n + K, trees)
    R, c, vl = 2, 1.25, 0.75
    cap_sims = 2 * sims
    keep = cap_sims + 1 if cap == "S" else cap
    b = _batch_with_roots(roots, n)
    b.set_stream_base(300)
    m = BatchedMCTS(b, trees, cap_sims, R, c, selection=kind, solve=solve, leaves_per_step=K, virtual_loss=vl)
    m.begin(0, trees)
    counter = _Counted()
    refs = [counter.wrap(make(kind, solve, r, 300 + t, R, c, K, vl)) for t, r in enumerate(roots)]
    rng = random.Random(n * 10 + K)
    b.stats_reset()
    m.run(sims)
    for ref in refs:
        spec_run(ref, sims, K)
    _assert_same(m, refs, n, "first search")
    for move, kept in enumerate((keep, sims + 1)):  # the second: what a capacity of 2*sims allows every move
        # categories t + 3*move: a ply-0 root advanced along its best move meets the swap next
        actions = np.asarray([choose(ref, n, t + 3 * move, rng) for t, ref in enumerate(refs)], dtype=np.int32)
        l0 = b.stats()["kernel_launches"]
        status = m.advance(actions, kept)
        assert b.stats()["kernel_launches"] - l0 == 1
        want = [reuse_spec.advance(ref, int(a), kept) for ref, a in zip(refs, actions)]
        assert status.tolist() == want, (move, actions.tolist())
        _assert_same(m, refs, n, ("advanced", move))
        m.run(sims)
        for ref in refs:
            spec_run(ref, sims, K)
        _assert_same(m, refs, n, ("continued", move))
    st = b.stats()
    assert (st["plies"], st["games"]) == (counter.plies, counter.games)


def _stepwise(m, b, refs, n, trees, K, steps):
    """The device search and the specification in lock step with stand-in values and priors: leaf records and
    statuses at every step."""
    rows = trees * K
    for step in range(steps):
        status = m.select(trees)
        leaves = b.export_state(trees, rows)
        values = np.stack([mcts_spec.stand_in_value(r) for r in leaves])
        priors = np.stack([puct_spec.stand_in_priors(r, n) for r in leaves])
        for t, ref in enumerate(refs):
            if K > 1:
                got = ref.select_step(K)
                for j, (leaf, term) in enumerate(got):
                    assert status[t * K + j] == int(term), (step, t, j)
                    assert np.array_equal(leaves[t * K + j], ref.nodes[leaf].state.export_record()), (step, t, j)
                ref.backup_step([None if term else values[t * K + j] for j, (_, term) in enumerate(got)],
                                [None if term else priors[t * K + j] for j, (_, term) in enumerate(got)])
                continue
            leaf, st = ref.select()
            assert status[t] == int(st), (step, t)
            if leaf is not None:
                assert np.array_equal(leaves[t], ref.nodes[leaf].state.export_record()), (step, t)
            if isinstance(ref, puct_spec.Search):
                ref.backup(None if st else values[t], None if st else priors[t])
            else:
                ref.backup(None if st else values[t])
        m.backup(values, priors if m.selection == "puct" else None)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,solve,K", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("n", [5, 8, 12, 24])
def test_stepwise_form_across_advances_matches_spec(oracle_mod, kind, solve, K, n):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    trees, sims = 12 if n < 24 else 6, 16
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 7 * n + K, trees)
    b = _batch_with_roots(roots, n, extra=trees * K)
    m = BatchedMCTS(b, trees, 2 * sims, 1, 2.0, selection=kind, solve=solve, leaves_per_step=K, virtual_loss=1.5)
    m.begin(0, trees)
    refs = [make(kind, solve, r, t, 1, 2.0, K, 1.5) for t, r in enumerate(roots)]
    rng = random.Random(n + K)
    _stepwise(m, b, refs, n, trees, K, sims // K)
    for move, keep in enumerate((2 * sims + 1, 3, 1, sims + 1)):
        actions = np.asarray([choose(ref, n, t + move, rng) for t, ref in enumerate(refs)], dtype=np.int32)
        status = m.advance(actions, keep)
        assert status.tolist() == [reuse_spec.advance(ref, int(a), keep) for ref, a in zip(refs, actions)]
        _stepwise(m, b, refs, n, trees, K, sims // K)
        _assert_same(m, refs, n, ("stepwise", move))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,solve,K", CASES, ids=CASE_IDS)
def test_chains_of_advances_over_whole_games(oracle_mod, kind, solve, K):
    """8 trees at n = 8 advance along their best move every move until every game is over."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 8, 24
    g = oracle_mod.OracleGame(n)
    roots = [g.new_initial_state() for _ in range(trees)]
    for t, r in enumerate(roots):
        for a in r.clone().playout_philox(SEED, 40 + t)[:t]:
            r.apply_action(a)
    b = _batch_with_roots(roots, n)
    m = BatchedMCTS(b, trees, 2 * sims, 1, 2.0, selection=kind, solve=solve, leaves_per_step=K)
    m.begin(0, trees)
    refs = [make(kind, solve, r, t, 1, 2.0, K) for t, r in enumerate(roots)]
    moves = 0
    while not all(root_state(ref).is_terminal() for ref in refs):
        m.run(sims)
        for ref in refs:
            spec_run(ref, sims, K)
        _assert_same(m, refs, n, moves)
        best = m.best()
        # a terminal root stays (-1); a finished solver tree without root edges plays its first legal move
        actions = np.asarray([-1 if root_state(ref).is_terminal() else
                              (int(a) if a >= 0 else root_state(ref).legal_actions()[0])
                              for ref, a in zip(refs, best)], dtype=np.int32)
        status = m.advance(actions, sims + 1)
        assert status.tolist() == [reuse_spec.advance(ref, int(a), sims + 1) for ref, a in zip(refs, actions)]
        moves += 1
        assert moves < n * n
    assert moves > 3


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uct", "puct"])
def test_host_and_device_pointers_give_the_same_trees(oracle_mod, kind):
    import torch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, ROOT_ILLEGAL
    n, trees, sims = 8, 16, 32
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 23, trees)
    b = _batch_with_roots(roots, n)
    b.use_torch_stream()
    refs = [make(kind, False, r, t) for t, r in enumerate(roots)]
    for ref in refs:
        spec_run(ref, sims, 1)
    rng = random.Random(2)
    actions = np.asarray([choose(ref, n, t, rng) for t, ref in enumerate(refs)], dtype=np.int32)
    out = []
    for device in (False, True):
        m = BatchedMCTS(b, trees, 2 * sims, 1, selection=kind)
        m.begin(0, trees)
        m.run(sims)
        if device:
            status = torch.full((trees,), 7, dtype=torch.int32, device="cuda")
            ret = m.advance(torch.from_numpy(actions).cuda(), 9, out_status=status)
            assert ret is status  # asynchronous: read after the stream
            torch.cuda.current_stream().synchronize()
            status = status.cpu().numpy()
        else:
            status = m.advance(actions, 9)
        assert ROOT_ILLEGAL not in status.tolist()
        m.run(sims)
        out.append((status, m.root_stats()))
        m.close()
    assert out[0][0].tolist() == out[1][0].tolist()
    for x, y in zip(out[0][1], out[1][1]):
        assert x.tobytes() == y.tobytes()
    # an illegal action with device statuses: the call returns, the status reports it
    m = BatchedMCTS(b, trees, 2 * sims, 1, selection=kind)
    m.begin(0, trees)
    bad = actions.copy()
    bad[3] = n * n + 5
    status = torch.zeros(trees, dtype=torch.int32, device="cuda")
    m.advance(torch.from_numpy(bad).cuda(), 9, out_status=status)
    torch.cuda.current_stream().synchronize()
    assert status.cpu().numpy()[3] == ROOT_ILLEGAL


@pytest.mark.gpu
def test_errors_leave_the_search_exact(oracle_mod):
    from twixt_for_open_spiel_b200.batch import SpielFatalError
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, ROOT_ILLEGAL
    n, trees, sims = 8, 6, 30
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 31, trees)  # tree 4 is terminal
    assert roots[4].is_terminal()
    b = _batch_with_roots(roots, n, extra=trees)
    m = BatchedMCTS(b, trees, sims, 2, selection="puct")
    with pytest.raises(ValueError, match="no search begun"):
        m.advance([0] * trees, 5)
    with pytest.raises(ValueError, match="no search begun"):
        m.set_root_priors(np.full((trees, n * n), 0.1, np.float32))
    m.begin(0, trees)
    refs = [make("puct", False, r, t, 2) for t, r in enumerate(roots)]
    m.run(10)
    for ref in refs:
        spec_run(ref, 10, 1)
    legal = [choose(ref, n, 0, random.Random(0)) for ref in refs]
    for keep in (0, -1, sims + 2):
        with pytest.raises(ValueError, match="keep_nodes"):
            m.advance(legal, keep)
    m.select(trees)
    with pytest.raises(ValueError, match="awaits its backup"):
        m.advance(legal, 5)
    with pytest.raises(ValueError, match="awaits its backup"):
        m.set_root_priors(np.full((trees, n * n), 0.1, np.float32))
    leaves = b.export_state(trees, trees)
    values = np.stack([mcts_spec.stand_in_value(r) for r in leaves])
    priors = np.stack([puct_spec.stand_in_priors(r, n) for r in leaves])
    m.backup(values, priors)
    for t, ref in enumerate(refs):
        leaf, term = ref.select()
        ref.backup(None if term else values[t], None if term else priors[t])
    # illegal actions: out of range, a move at the terminal root, -2; the tree is unchanged, the others advance
    for bad_tree, bad_action in ((1, n * n), (4, 0), (2, -2)):
        acts = list(legal)
        acts[bad_tree] = bad_action
        l0 = b.stats()["kernel_launches"]
        with pytest.raises(SpielFatalError, match="Not a legal action: %d$" % bad_action):
            m.advance(acts, sims + 1)
        assert b.stats()["kernel_launches"] - l0 == 1
        got = [reuse_spec.advance(ref, a, sims + 1) for ref, a in zip(refs, acts)]
        assert [t for t, x in enumerate(got) if x == ROOT_ILLEGAL] == [bad_tree]
        _assert_same(m, refs, n, ("illegal", bad_tree))
        legal = [-1] * trees
    m.run(4)
    for ref in refs:
        spec_run(ref, 4, 1)
    _assert_same(m, refs, n, "after errors")
    # the budget: after an advance to keep nodes a tree takes at most S - keep more simulations
    m.begin(0, trees)
    m.run(sims)
    m.advance([-1] * trees, 20)
    with pytest.raises(ValueError, match="node slots"):
        m.run(sims + 1 - 20 + 1)
    m.run(sims + 1 - 20)
    with pytest.raises(ValueError, match="node slots"):
        m.run(1)
    uct = BatchedMCTS(b, trees, sims, 2)
    uct.begin(0, trees)
    with pytest.raises(ValueError, match="not a PUCT search"):
        uct.set_root_priors(np.full((trees, n * n), 0.1, np.float32))
    with pytest.raises(ValueError, match="31 simulations since begin would exceed max_simulations 30"):
        uct.run(sims + 1)  # without an advance: the check and its text as before


@pytest.mark.gpu
def test_rollout_counter_check_and_ln_table_growth(oracle_mod):
    """The simulation counter carries on across advances: k*R + r must stay below 2^32.  N(root) outgrows the S
    entries of the ln table at n = 5 when trees are kept over many moves; the grown table gives the spec's
    scores."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n = 5
    g = oracle_mod.OracleGame(n)
    root = g.new_initial_state()
    b = _batch_with_roots([root], n, extra=1)
    R = 1 << 24
    m = BatchedMCTS(b, 1, 255, R)
    m.begin(0, 1)
    v = np.asarray([[0.25, -0.25]], dtype=np.float32)
    for _ in range(255):
        m.select(1)
        m.backup(v)
    m.advance([-1], 1)
    m.select(1)
    m.backup(v)  # k = 255: (255 + 1) * R = 2^32, the last counter that fits
    m.advance([-1], 1)
    with pytest.raises(ValueError, match="2\\^32"):
        m.select(1)
    m.close()
    # UCT at n = 5 with capacity 40: N(root) passes S = 41 after a few -1 advances, then real moves
    roots = mcts_spec.root_positions(g, n, 3, 6)
    b = _batch_with_roots(roots, n)
    m = BatchedMCTS(b, 6, 40, 1, 1.0)
    m.begin(0, 6)
    refs = [make("uct", False, r, t, 1, 1.0) for t, r in enumerate(roots)]
    rng = random.Random(4)
    for move in range(14):
        m.run(20)
        for ref in refs:
            spec_run(ref, 20, 1)
        _assert_same(m, refs, n, move)
        acts = [-1 if move < 8 else choose(ref, n, 0, rng) for ref in refs]
        if move == 7:
            assert max(ref.nodes[0].n for ref in refs) > 41  # past the arena's ln table
        status = m.advance(acts, 21)
        assert status.tolist() == [reuse_spec.advance(ref, a, 21) for ref, a in zip(refs, acts)]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 4])
def test_set_root_priors_matches_spec_and_skips_fresh_roots(oracle_mod, K):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, ROOT_FRESH, ROOT_KEPT
    n, trees, sims = 8, 12, 32
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 41, trees)
    b = _batch_with_roots(roots, n, extra=trees * K)
    m = BatchedMCTS(b, trees, 2 * sims, 1, selection="puct", leaves_per_step=K)
    m.begin(0, trees)
    refs = [make("puct", False, r, t, K=K) for t, r in enumerate(roots)]
    _stepwise(m, b, refs, n, trees, K, sims // K)
    rng = random.Random(9)
    actions = np.asarray([choose(ref, n, t, rng) for t, ref in enumerate(refs)], dtype=np.int32)
    status = m.advance(actions, sims + 1)
    for ref, a in zip(refs, actions):
        reuse_spec.advance(ref, int(a), sims + 1)
    noisy = np.random.default_rng(3).random((trees, n * n)).astype(np.float32)
    l0 = b.stats()["kernel_launches"]
    m.set_root_priors(noisy)
    assert b.stats()["kernel_launches"] - l0 == 1
    for t, ref in enumerate(refs):
        for c in ref.nodes[0].children:  # only expanded roots have children
            c.prior = float(noisy[t, c.action])
    assert ROOT_FRESH in status.tolist() and ROOT_KEPT in status.tolist()
    _stepwise(m, b, refs, n, trees, K, sims // K)
    _assert_same(m, refs, n, "after set_root_priors")


@pytest.mark.gpu
def test_bot_with_tree_reuse_plays_the_spec_moves(oracle_mod):
    from twixt_for_open_spiel_b200 import load_game
    from twixt_for_open_spiel_b200.mcts import MCTSBot
    n, sims, R, c, seed = 8, 60, 2, 2.0, 5
    game = load_game("twixt(board_size=%d)" % n)
    bot = MCTSBot(game, uct_c=c, max_simulations=sims, n_rollouts=R, seed=seed, reuse_tree=True)
    g = oracle_mod.OracleGame(n)
    state, ostate = game.new_initial_state(), g.new_initial_state()
    ref = None
    history, searched = [], 0  # the actions played, and how many of them the specification's root holds
    rng = random.Random(8)
    try:
        while not state.is_terminal():
            a = bot.step(state)
            if ref is None:
                ref = mcts_spec.Search(ostate, seed, 0, R, c)
            else:
                for x in history[searched:]:
                    reuse_spec.advance(ref, x, sims + 1)
            searched = len(history)
            ref.run(sims)
            assert a == ref.root_stats(n)[2]
            assert a in state.legal_actions()
            state.apply_action(a)
            ostate.apply_action(a)
            history.append(a)
            if not state.is_terminal():  # the opponent: a random move
                b = rng.choice(state.legal_actions())
                state.apply_action(b)
                ostate.apply_action(b)
                history.append(b)
    finally:
        bot.close()


@pytest.mark.gpu
def test_self_play_example_with_tree_reuse_runs_to_the_end():
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    try:
        import alphazero_selfplay
    finally:
        sys.path.pop(0)
    for K in (1, 2):
        traj, returns = alphazero_selfplay.self_play(n=6, games=8, sims=8, verbose=False, leaves_per_step=K,
                                                     reuse_tree=True)
        assert len(traj) == 8 and all(len(t) > 0 for t in traj)
        assert returns.shape == (8, 2)


@pytest.mark.gpu
def test_advance_at_scale(oracle_mod):
    """8 192 PUCT trees at n = 12 after a 400-simulation search, advanced along their best move with keep 401; the
    kept root statistics of a sample of trees are checked against the specification, and the kept visit counts of
    all of them against the root statistics before the advance."""
    import torch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, ROOT_KEPT
    n, trees, sims = 12, 8192, 400
    g = oracle_mod.OracleGame(n)
    roots = []
    for t in range(trees):
        st = g.new_initial_state()
        for a in st.clone().playout_philox(SEED, t)[:t % 11]:
            st.apply_action(a)
        roots.append(st)
    b = _batch_with_roots(roots, n)
    b.use_torch_stream()
    m = BatchedMCTS(b, trees, 2 * sims, 1, selection="puct")
    m.begin(0, trees)
    m.run(sims)
    before, _, best = m.root_stats()
    l0 = b.stats()["kernel_launches"]
    status = torch.zeros(trees, dtype=torch.int32, device="cuda")
    m.advance(torch.from_numpy(best).cuda(), sims + 1, out_status=status)
    torch.cuda.current_stream().synchronize()
    assert b.stats()["kernel_launches"] - l0 == 1
    assert (status.cpu().numpy() == ROOT_KEPT).all()
    visits, sums, best2 = m.root_stats()
    # N(new root) = N(a) of the move played, one of which evaluated the new root itself
    assert np.array_equal(visits.sum(axis=1), before[np.arange(trees), best] - 1)
    for t in (5, trees - 2):
        ref = make("puct", False, roots[t], t).run(sims)
        assert reuse_spec.advance(ref, int(best[t]), sims + 1) == ROOT_KEPT
        v, w, bb = ref.root_stats(n)
        assert np.array_equal(visits[t], v) and sums[t].tobytes() == w.tobytes() and best2[t] == bb, t
