"""Batched MCTS (twixt_mcts_*, twixt_for_open_spiel_b200/mcts.py) against its executable specification
tests/mcts_spec.py.  CPU: the specification's own properties, the product's search helpers compiled for the
host (tests/mcts_harness.cc) running complete searches node for node against it, and the score's bit
exactness.  GPU: the device search bit for bit against the specification, the stepwise form, reproducibility,
host / device paths, errors, the bot and a search at scale."""
import ctypes as C
import math
import os
import random
import subprocess

import numpy as np
import pytest

import mcts_spec as spec

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "twixt_for_open_spiel_b200", "csrc")
SEED = 0x6D637473


def P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def mh():
    out_dir = os.path.join(HERE, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libmctsharness.so")
    src = os.path.join(HERE, "mcts_harness.cc")
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-x", "c++", "-fPIC",
                               "-shared", "-I", CSRC, "-o", so, src])
    lib = C.CDLL(so)
    lib.mh_score.restype = C.c_double
    lib.mh_score.argtypes = [C.c_double, C.c_uint32, C.c_double, C.c_double]
    lib.mh_draw.restype = C.c_uint32
    lib.mh_draw.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
    lib.mh_bytes_per_tree.restype = C.c_int64
    lib.mh_bytes_per_tree.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.mh_search.restype = C.c_int
    lib.mh_search.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_double, C.c_int] + \
        [C.c_void_p] * 7
    return lib


def harness_search(mh, root, n, seed, T, R, c, sims):
    S, M = sims + 1, n * (n - 2)
    parent = np.zeros(S, dtype=np.int32)
    action = np.zeros(S, dtype=np.int32)
    visits = np.zeros(S, dtype=np.uint32)
    legal = np.zeros(S, dtype=np.int32)
    en = np.zeros((S, M), dtype=np.uint32)
    ew = np.zeros((S, M), dtype=np.float64)
    best = np.zeros(1, dtype=np.int32)
    rec = np.ascontiguousarray(root.export_record())
    count = mh.mh_search(P(rec), n, seed, T, R, c, sims, P(parent), P(action), P(visits), P(legal), P(en), P(ew),
                         P(best))
    return count, parent, action, visits, legal, en, ew, int(best[0])


def one_move_root(game, n):
    """A position whose player to move has exactly one legal action."""
    for s in range(5000):
        st = game.new_initial_state()
        for a in st.clone().playout_philox(SEED, s):
            st.apply_action(a)
            if not st.is_terminal() and len(st.legal_actions()) == 1:
                return st
    raise AssertionError("no one-move position found")


# ------------------------------------------------------------------------------- the specification itself ---
def test_spec_root_visits_and_order(oracle_mod):
    g = oracle_mod.OracleGame(5)
    s = spec.Search(g.new_initial_state(), SEED, 7, n_rollouts=2)
    L = len(g.new_initial_state().legal_actions())
    for k in range(1, 60):
        s.simulate()
        root = s.nodes[0]
        assert sum(root.edge_n) == k - 1 and root.n == k
        if k - 1 <= L:  # every edge once before any twice
            assert max(root.edge_n or [0]) <= 1
    assert min(s.nodes[0].edge_n) >= 1


def test_spec_swap_edge_terminal_and_single_move(oracle_mod):
    g = oracle_mod.OracleGame(6)
    st = g.new_initial_state()
    st.apply_action(13)
    s = spec.Search(st, SEED, 3).run(30)
    assert 13 in s.nodes[0].actions  # the swap offer is an edge at ply 1
    term = g.new_initial_state()
    for a in term.clone().playout_philox(SEED, 5):
        term.apply_action(a)
    assert term.is_terminal()
    s = spec.Search(term, SEED, 4).run(10)
    v, w, best = s.root_stats(6)
    assert v.sum() == 0 and best == -1 and s.nodes[0].n == 10 and len(s.nodes) == 1
    g5 = oracle_mod.OracleGame(5)
    one = one_move_root(g5, 5)
    s = spec.Search(one, SEED, 9, n_rollouts=3).run(12)
    v, w, best = s.root_stats(5)
    assert best == one.legal_actions()[0] and v.sum() == 11


def test_spec_hand_traced_four_simulations(oracle_mod):
    """n = 5, R = 1: simulation 0 evaluates the root, 1..3 each take the drawn unvisited root edge."""
    g = oracle_mod.OracleGame(5)
    root = g.new_initial_state()
    T = 11
    s = spec.Search(root, SEED, T, n_rollouts=1).run(4)
    legal = root.legal_actions()
    unvisited = list(legal)
    expect = {}
    for k in (1, 2, 3):
        w = oracle_mod.philox([T, 0, k, 1], [SEED & 0xFFFFFFFF, SEED >> 32])[0]
        a = unvisited.pop((w * len(unvisited)) >> 32)
        child = root.clone()
        child.apply_action(a)
        child.playout_philox(SEED, (T << 32) | k)
        expect[a] = child.returns()[0]  # red is to move at the root
    v, sums, best = s.root_stats(5)
    assert {a: int(v[a]) for a in np.nonzero(v)[0]} == {a: 1 for a in expect}
    assert {a: float(sums[a]) for a in expect} == expect
    assert s.nodes[0].n == 4 and len(s.nodes) == 4
    top = max(expect.items(), key=lambda kv: (kv[1], -kv[0]))[0]
    assert best == top


# ----------------------------------------------------------------------- host harness vs specification ---
@pytest.mark.parametrize("n", [5, 8, 12])
def test_harness_matches_spec_node_for_node(mh, oracle_mod, n):
    g = oracle_mod.OracleGame(n)
    roots = spec.root_positions(g, n, 40 + n, 6)
    sims_for = {5: 200, 8: 120, 12: 60}
    for i, root in enumerate(roots):
        R = 1 if i % 2 == 0 else 3
        sims = sims_for[n] if i % 3 != 2 else 37
        c = 2.0 if i % 2 == 0 else 0.7
        T = 1000 * n + i
        ref = spec.Search(root, SEED, T, R, c).run(sims)
        count, parent, action, visits, legal, en, ew, best = harness_search(mh, root, n, SEED, T, R, c, sims)
        assert count == len(ref.nodes), (n, i)
        for k, node in enumerate(ref.nodes):
            assert (parent[k], action[k], visits[k]) == (node.parent, node.action, node.n), (n, i, k)
            L = -1 if node.actions is None else len(node.actions)
            assert legal[k] == L, (n, i, k)
            if L > 0:
                assert en[k, :L].tolist() == node.edge_n, (n, i, k)
                assert ew[k, :L].tobytes() == np.asarray(node.edge_w, dtype=np.float64).tobytes(), (n, i, k)
        assert best == ref.root_stats(n)[2], (n, i)


def test_score_is_bit_exact_on_the_host(mh):
    rng = random.Random(5)
    for _ in range(100000):
        n = rng.randrange(1, 5000)
        parent = rng.randrange(max(n, 1), 10001)
        w = rng.uniform(-n, n) if rng.random() < 0.7 else float(rng.randrange(-n, n + 1)) / rng.choice((1, 2, 3, 4))
        c = rng.choice((2.0, 1.4142135623730951, 0.5, 0.0, rng.uniform(0, 10)))
        expect = w / n + c * math.sqrt(math.log(parent) / n)
        got = mh.mh_score(w, n, math.log(parent), c)
        assert got.hex() == expect.hex(), (w, n, parent, c)


def test_draw_and_bytes_per_tree(mh, oracle_mod):
    for k in range(200):
        U = 1 + (k * 37) % 500
        assert mh.mh_draw(SEED, 77, k, U) == spec.draw(SEED, 77, k, U)
    # at n = 12: (400 + 1) node slots of 448 + 8 + 18 * 120 bytes, 16 + 8 * (141 + 1) path bytes (the longest
    # game has 141 moves), 4 rollout slots of 448 + 16 bytes
    assert mh.mh_bytes_per_tree(12, 400, 4) == 401 * (448 + 8 + 2160) + 16 + 8 * 142 + 4 * (448 + 16)


# ---------------------------------------------------------------------------------------------- GPU ---
def _batch_with_roots(roots, n, seed=SEED, extra=0):
    from twixt_for_open_spiel_b200 import TwixTBatch
    b = TwixTBatch(n, len(roots) + extra, 0, seed)
    b.import_state(np.stack([r.export_record() for r in roots]), 0)
    return b


def _assert_stats_equal(got, refs, n, tag):
    visits, sums, best = got
    for t, ref in enumerate(refs):
        v, w, bst = ref.root_stats(n)
        assert np.array_equal(visits[t], v), (tag, t)
        assert sums[t].tobytes() == w.tobytes(), (tag, t)
        assert best[t] == bst, (tag, t)


@pytest.mark.gpu
@pytest.mark.parametrize("n,trees,sims,R", [(5, 48, 300, 4), (8, 48, 200, 1), (12, 32, 120, 4), (24, 32, 50, 1),
                                            (24, 32, 50, 4)])
def test_device_search_matches_spec(oracle_mod, n, trees, sims, R):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = spec.root_positions(g, n, 7 * n + R, trees)
    b = _batch_with_roots(roots, n)
    b.set_stream_base(100)
    m = BatchedMCTS(b, trees, sims, R, 1.5)
    m.begin(0, trees)
    m.run(sims)
    refs = [spec.Search(r, SEED, 100 + t, R, 1.5).run(sims) for t, r in enumerate(roots)]
    _assert_stats_equal(m.root_stats(), refs, n, (n, R))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5, 12])
def test_stepwise_form_matches_spec(oracle_mod, n):
    from twixt_for_open_spiel_b200.mcts import LEAF_NEEDS_VALUE, LEAF_TERMINAL, BatchedMCTS
    trees, sims = 24, 60
    g = oracle_mod.OracleGame(n)
    roots = spec.root_positions(g, n, 3 * n, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    m = BatchedMCTS(b, trees, sims, 1)
    m.begin(0, trees)
    refs = [spec.Search(r, SEED, t, 1, 2.0) for t, r in enumerate(roots)]
    for k in range(sims):
        status = m.select(trees)
        leaves = b.export_state(trees, trees)
        values = np.zeros((trees, 2), dtype=np.float32)
        for t, ref in enumerate(refs):
            leaf, terminal = ref.select()
            assert np.array_equal(leaves[t], ref.nodes[leaf].state.export_record()), (n, k, t)
            assert status[t] == (LEAF_TERMINAL if terminal else LEAF_NEEDS_VALUE), (n, k, t)
            values[t] = spec.stand_in_value(leaves[t])
            ref.backup(values[t])
        m.backup(values)
    _assert_stats_equal(m.root_stats(), refs, n, n)


@pytest.mark.gpu
def test_reproducibility(oracle_mod):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n = 8
    g = oracle_mod.OracleGame(n)
    roots = spec.root_positions(g, n, 99, 64)
    b = _batch_with_roots(roots, n)
    before = b.export_state()
    m1 = BatchedMCTS(b, 64, 200, 2)
    m1.begin(0, 64)
    m1.run(100)
    m1.run(100)
    split = m1.root_stats()
    m2 = BatchedMCTS(b, 64, 200, 2)
    m2.begin(0, 64)
    m2.run(200)
    whole = m2.root_stats()
    for x, y in zip(split, whole):
        assert x.tobytes() == y.tobytes()
    halves = []
    m3 = BatchedMCTS(b, 32, 200, 2)
    for first in (0, 32):
        m3.begin(first, 32)
        m3.run(200)
        halves.append(m3.root_stats())
    for i in range(3):
        assert np.concatenate([halves[0][i], halves[1][i]]).tobytes() == whole[i].tobytes()
    assert b.export_state().tobytes() == before.tobytes()


@pytest.mark.gpu
def test_device_tensors_launch_count_and_errors(oracle_mod):
    import torch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees = 8, 16
    g = oracle_mod.OracleGame(n)
    roots = spec.root_positions(g, n, 5, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    m = BatchedMCTS(b, trees, 40, 2)
    m.begin(0, trees)
    l0 = b.stats()["kernel_launches"]
    m.run(20)
    assert b.stats()["kernel_launches"] - l0 <= 3 * 20
    host = m.root_stats()
    dev = (torch.zeros((trees, n * n), dtype=torch.int32, device="cuda"),
           torch.zeros((trees, n * n), dtype=torch.float64, device="cuda"),
           torch.zeros(trees, dtype=torch.int32, device="cuda"))
    m.root_stats(*dev)
    b.synchronize()
    for x, y in zip(host, dev):
        assert x.tobytes() == y.cpu().numpy().tobytes()
    # stepwise with device values and statuses equals the host path
    m2 = BatchedMCTS(b, trees, 40, 2)
    m2.begin(0, trees)
    m2.run(20)
    for _ in range(5):
        st_h = m.select(trees)
        vals = np.stack([spec.stand_in_value(r) for r in b.export_state(trees, trees)])
        m.backup(vals)
        st_d = torch.zeros(trees, dtype=torch.int32, device="cuda")
        m2.select(trees, st_d)
        m2.backup(torch.from_numpy(vals).cuda())
        b.synchronize()
        assert np.array_equal(st_h, st_d.cpu().numpy())
    for x, y in zip(m.root_stats(), m2.root_stats()):
        assert x.tobytes() == y.tobytes()
    # every argument error leaves the trees unchanged
    snap = m.root_stats()
    vals = np.zeros((trees, 2), dtype=np.float32)
    bad_calls = [
        lambda: m.begin(0, trees + 1),
        lambda: m.begin(b.num_envs - 2, 4),
        lambda: m.run(16),                      # 25 + 16 > 40
        lambda: m.select(b.num_envs - 1),
        lambda: m.backup(vals),                 # no select pending
    ]
    for call in bad_calls:
        with pytest.raises(ValueError):
            call()
        for x, y in zip(snap, m.root_stats()):
            assert x.tobytes() == y.tobytes()
    m.select(trees)
    for call in (lambda: m.select(trees), lambda: m.run(1)):
        with pytest.raises(ValueError):
            call()
    m.backup(vals)
    b.set_stream_base((1 << 32) - 4)
    with pytest.raises(ValueError):
        m.begin(0, trees)
    b.set_stream_base(0)
    for c in (float("nan"), float("inf"), -1.0):
        with pytest.raises(ValueError):
            BatchedMCTS(b, trees, 40, 2, c)
    with pytest.raises(ValueError):
        BatchedMCTS(b, 1, 1 << 30, 8)  # max_simulations * n_rollouts >= 2^32
    with pytest.raises(MemoryError, match="bytes per tree"):
        BatchedMCTS(b, 1 << 40, 1000, 1)
    for x, y in zip(snap[:2], m.root_stats()[:2]):
        assert x.shape == y.shape


@pytest.mark.gpu
def test_bot_matches_batched_search_and_plays_a_game(oracle_mod):
    from twixt_for_open_spiel_b200 import TwixTBatch, load_game
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, MCTSBot
    game = load_game("twixt(board_size=8)")
    bot = MCTSBot(game, uct_c=2.0, max_simulations=200, n_rollouts=4, seed=3)
    state = game.new_initial_state()
    state.apply_action(10)
    a = bot.step(state)
    assert a in state.legal_actions()
    b = TwixTBatch(8, 1, 0, 3)
    b.import_state(state.export_record(), 0)
    m = BatchedMCTS(b, 1, 200, 4, 2.0)
    m.begin(0, 1)
    m.run(200)
    assert int(m.best()[0]) == a
    og = oracle_mod.OracleGame(8)
    ost = og.new_initial_state()
    ost.apply_action(10)
    assert spec.Search(ost, 3, 0, 4, 2.0).run(200).root_stats(8)[2] == a
    rng = random.Random(17)
    state = game.new_initial_state()
    bot = MCTSBot(game, max_simulations=100, n_rollouts=4, seed=1)
    while not state.is_terminal():
        if state.current_player() == 0:
            act = bot.step(state)
        else:
            act = rng.choice(state.legal_actions())
        assert act in state.legal_actions()
        state.apply_action(act)
    assert sorted(state.returns()) in ([-1.0, 1.0], [0.0, 0.0])


@pytest.mark.gpu
def test_search_at_scale(oracle_mod):
    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims, R = 12, 8192, 100, 4
    b = TwixTBatch(n, trees, 0, SEED)
    group = trees // 8
    for gi in range(8):
        b.playout(gi * group, group, max_plies=3 * gi, want_returns=False, want_lengths=False)
    m = BatchedMCTS(b, trees, sims, R)
    m.begin(0, trees)
    m.run(sims)
    visits, sums, best = m.root_stats()
    g = oracle_mod.OracleGame(n)
    recs = b.export_state()
    for t in random.Random(8).sample(range(trees), 16):
        root = g.new_initial_state()
        for a in root.clone().playout_philox(SEED, t, 3 * (t // group)):
            root.apply_action(a)
        assert np.array_equal(root.export_record(), recs[t])
        ref = spec.Search(root, SEED, t, R, 2.0).run(sims)
        v, w, bst = ref.root_stats(n)
        assert np.array_equal(visits[t], v) and sums[t].tobytes() == w.tobytes() and best[t] == bst, t
