"""PUCT search with policy priors (twixt_mcts_create_puct, twixt_mcts_backup_priors, BatchedMCTS(selection=
"puct")) against its executable specification tests/puct_spec.py.  CPU: the specification's own properties, the
product's helpers compiled for the host (tests/puct_harness.cc) running searches node for node against it, the
score's bit exactness and add_dirichlet_noise.  GPU: the device search bit for bit against the specification
(built-in rollouts and the stepwise form), host / device paths, reproducibility, launch counts, errors, the
self-play example and a search at scale."""
import ctypes as C
import math
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import mcts_spec
import puct_spec as spec

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "twixt_for_open_spiel_b200", "csrc")
SEED = 0x70756374


def P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def ph():
    out_dir = os.path.join(HERE, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libpuctharness.so")
    src = os.path.join(HERE, "puct_harness.cc")
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-x", "c++", "-fPIC",
                               "-shared", "-I", CSRC, "-o", so, src])
    lib = C.CDLL(so)
    lib.ph_score.restype = C.c_double
    lib.ph_score.argtypes = [C.c_double, C.c_uint32, C.c_float, C.c_uint32, C.c_double]
    lib.ph_tie_key.restype = C.c_uint32
    lib.ph_tie_key.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
    lib.ph_bytes_per_tree.restype = C.c_int64
    lib.ph_bytes_per_tree.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.ph_create.restype = C.c_void_p
    lib.ph_create.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_double, C.c_int]
    lib.ph_destroy.argtypes = [C.c_void_p]
    lib.ph_select.restype = C.c_int
    lib.ph_select.argtypes = [C.c_void_p, C.c_void_p]
    lib.ph_backup.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ph_dump.restype = C.c_int
    lib.ph_dump.argtypes = [C.c_void_p] + [C.c_void_p] * 8
    return lib


def zero_value(record):
    return np.zeros(2, dtype=np.float32)


def harness_search(ph, root, n, seed, T, R, c, sims, value_fn=None, prior_fn=None):
    """A complete search on the host harness; value_fn / prior_fn None: host rollouts / uniform priors."""
    rec = np.ascontiguousarray(root.export_record())
    h = ph.ph_create(P(rec), n, seed, T, R, c, sims)
    leaf = np.zeros_like(rec)
    try:
        for _ in range(sims):
            terminal = ph.ph_select(h, P(leaf))
            vals = pri = None
            if not terminal and value_fn is not None:
                vals = np.ascontiguousarray(value_fn(leaf), dtype=np.float32)
            if not terminal and prior_fn is not None:
                pri = np.ascontiguousarray(prior_fn(leaf), dtype=np.float32)
            ph.ph_backup(h, None if vals is None else P(vals), None if pri is None else P(pri))
        S, M = sims + 1, n * (n - 2)
        parent, action, legal = (np.zeros(S, dtype=np.int32) for _ in range(3))
        visits = np.zeros(S, dtype=np.uint32)
        en = np.zeros((S, M), dtype=np.uint32)
        ew = np.zeros((S, M), dtype=np.float64)
        ep = np.zeros((S, M), dtype=np.float32)
        best = np.zeros(1, dtype=np.int32)
        count = ph.ph_dump(h, P(parent), P(action), P(visits), P(legal), P(en), P(ew), P(ep), P(best))
    finally:
        ph.ph_destroy(h)
    return count, parent, action, visits, legal, en, ew, ep, int(best[0])


def assert_harness_matches(got, ref, n, tag):
    count, parent, action, visits, legal, en, ew, ep, best = got
    dump = ref.dump()
    assert count == len(dump), tag
    for k, (par, act, nn, L, e_n, e_w, e_p) in enumerate(dump):
        assert (parent[k], action[k], visits[k], legal[k]) == (par, act, nn, L), (tag, k)
        if L > 0:
            assert en[k, :L].tolist() == e_n, (tag, k)
            assert ew[k, :L].tobytes() == np.asarray(e_w, dtype=np.float64).tobytes(), (tag, k)
            assert ep[k, :L].tobytes() == np.asarray(e_p, dtype=np.float32).tobytes(), (tag, k)
    assert best == ref.root_stats(n)[2], tag


def winning_root(game, n):
    """A position whose player to move wins with one of its legal actions; returns (state, winning action)."""
    for s in range(5000):
        st = game.new_initial_state()
        acts = st.clone().playout_philox(SEED, s)
        for a in acts[:-1]:
            st.apply_action(a)
        mover = st.current_player()
        end = st.clone()
        end.apply_action(acts[-1])
        if end.returns()[mover] == 1.0:
            return st, acts[-1]
    raise AssertionError("no position one move from a win found")


# ------------------------------------------------------------------------------- the specification itself ---
def test_spec_uniform_priors_visit_root_edges_in_tie_key_order(oracle_mod):
    """n = 5, zero values: simulation 0 expands the root; every edge then scores c*P*sqrt(N(s)) while unvisited
    and half that once visited, so simulations 1.. take the root edges in ascending tie-key order."""
    g = oracle_mod.OracleGame(5)
    root = g.new_initial_state()
    T, sims = 11, 12
    s = spec.Search(root, SEED, T).run(sims, value_fn=zero_value)
    legal = root.legal_actions()
    keys = [oracle_mod.philox([T, 0, i, 2], [SEED & 0xFFFFFFFF, SEED >> 32])[0] for i in range(len(legal))]
    order = [legal[i] for i in sorted(range(len(legal)), key=lambda i: (keys[i], i))]
    assert [s.nodes[k].action for k in range(1, sims)] == order[:sims - 1]
    assert all(s.nodes[k].parent_slot == 0 for k in range(1, sims))
    v, _, best = s.root_stats(5)
    assert v.sum() == sims - 1 and best == order[0]  # all (0, 1, 0.0): the first in shuffled order


def test_spec_ignores_illegal_prior_entries(oracle_mod):
    """Changing every prior entry off the leaf's legal list changes nothing, bit for bit."""
    n = 6
    g = oracle_mod.OracleGame(n)
    root = mcts_spec.root_positions(g, n, 3, 3)[2]
    legal_of = {}

    def prior(rec, junk):
        p = spec.stand_in_priors(rec, n).copy()
        key = rec.tobytes()
        if junk:
            mask = np.ones(n * n, dtype=bool)
            mask[legal_of[key]] = False
            p[mask] = np.float32(junk)
        return p

    s0 = spec.Search(root, SEED, 1)
    s1 = spec.Search(root, SEED, 1)
    for _ in range(80):
        l0, t0 = s0.select()
        l1, t1 = s1.select()
        assert (l0, t0) == (l1, t1)
        st = s0.nodes[l0].state
        rec = st.export_record()
        legal_of[rec.tobytes()] = st.legal_actions() if not t0 else []
        v = mcts_spec.stand_in_value(rec)
        s0.backup(v, prior(rec, 0))
        s1.backup(v, prior(rec, 3.5))
    assert repr(s0.dump()) == repr(s1.dump())  # W as repr: bit for bit


def test_spec_concentrated_prior_draws_most_root_visits(oracle_mod):
    n = 8
    g = oracle_mod.OracleGame(n)
    root = g.new_initial_state()
    root.apply_action(20)
    legal = root.legal_actions()
    target = legal[len(legal) // 3]
    root_rec = root.export_record()

    def prior(rec):
        p = spec.stand_in_priors(rec, n)
        if np.array_equal(rec, root_rec):
            p = np.full(n * n, 0.01 / len(legal), dtype=np.float32)
            p[target] = 0.99
        return p

    s = spec.Search(root, SEED, 2, n_rollouts=1).run(200, None, prior)
    v, _, best = s.root_stats(n)
    assert v[target] > 0.5 * v.sum() and best == target


def test_spec_winning_edge_is_best_once_visited_and_scored_by_its_outcome(oracle_mod):
    n = 6
    g = oracle_mod.OracleGame(n)
    root, win = winning_root(g, n)
    s = spec.Search(root, SEED, 4, n_rollouts=1)
    seen = False
    for _ in range(150):
        s.simulate(None, lambda rec: spec.stand_in_priors(rec, n))
        child = next((c for c in s.nodes[0].children if c.action == win), None)
        if child is not None and child.explore_count > 0:
            seen = True
            assert child.outcome is not None and child.puct_value(s.nodes[0].explore_count, s.c) == 1.0
            assert s.root_stats(n)[2] == win
    assert seen


def test_spec_terminal_root(oracle_mod):
    g = oracle_mod.OracleGame(6)
    term = g.new_initial_state()
    for a in term.clone().playout_philox(SEED, 5):
        term.apply_action(a)
    s = spec.Search(term, SEED, 4).run(10, None, lambda rec: spec.stand_in_priors(rec, 6))
    v, w, best = s.root_stats(6)
    assert v.sum() == 0 and best == -1 and s.nodes[0].explore_count == 10 and len(s.nodes) == 1


# ----------------------------------------------------------------------- host harness vs specification ---
@pytest.mark.parametrize("n", [5, 8, 12])
def test_harness_matches_spec_node_for_node(ph, oracle_mod, n):
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 50 + n, 6)
    sims_for = {5: 150, 8: 100, 12: 50}
    prior = lambda rec: spec.stand_in_priors(rec, n)  # noqa: E731
    for i, root in enumerate(roots):
        R = 1 if i % 2 == 0 else 3
        c = 2.0 if i % 2 == 0 else 0.7
        T = 1000 * n + i
        sims = sims_for[n]
        # uniform priors + host rollouts
        ref = spec.Search(root, SEED, T, R, c).run(sims)
        assert_harness_matches(harness_search(ph, root, n, SEED, T, R, c, sims), ref, n, (n, i, "rollouts"))
        # stand-in priors and values
        ref = spec.Search(root, SEED, T, 1, c).run(sims, mcts_spec.stand_in_value, prior)
        got = harness_search(ph, root, n, SEED, T, 1, c, sims, mcts_spec.stand_in_value, prior)
        assert_harness_matches(got, ref, n, (n, i, "stand-in"))


def test_puct_score_is_bit_exact_on_the_host(ph):
    rng = random.Random(6)
    for _ in range(100000):
        na = rng.randrange(0, 5000) if rng.random() < 0.8 else 0
        ns = rng.randrange(max(na, 1), 10001)
        w = rng.uniform(-na, na) if rng.random() < 0.7 else float(rng.randrange(-na, na + 1)) / rng.choice((1, 2, 3))
        p = float(np.float32(rng.choice((rng.random(), 1.0 / rng.randrange(1, 600), 0.0, 1.0))))
        c = rng.choice((2.0, 1.25, 0.5, 0.0, rng.uniform(0, 10)))
        expect = (na and w / na) + c * p * math.sqrt(ns) / (na + 1)
        got = ph.ph_score(w, na, p, ns, c)
        assert got.hex() == float(expect).hex(), (w, na, p, ns, c)


def test_tie_key_and_bytes_per_tree(ph, oracle_mod):
    for k in range(200):
        T, slot, edge = 77 + k * 1013, (k * 37) % 401, (k * 11) % 528
        assert ph.ph_tie_key(SEED, T, slot, edge) == spec.tie_key(SEED, T, slot, edge)
    # at n = 12: (400 + 1) node slots of 448 + 8 + 27 * 120 bytes, 16 + 8 * (141 + 1) path bytes, 4 rollout slots
    # of 448 + 16 bytes
    assert ph.ph_bytes_per_tree(12, 400, 4) == 401 * (448 + 8 + 27 * 120) + 16 + 8 * 142 + 4 * (448 + 16)


def test_add_dirichlet_noise_on_cpu_tensors():
    import torch
    from twixt_for_open_spiel_b200.mcts import add_dirichlet_noise
    B, A = 64, 64
    gen = np.random.default_rng(0)
    mask = torch.from_numpy(gen.random((B, A)) < 0.6)
    mask[0] = False
    mask[1] = False
    mask[1, 7] = True
    p = torch.from_numpy(gen.random((B, A)).astype(np.float32))
    p = torch.where(mask, p, torch.full_like(p, 3.0))
    eps, alpha = 0.25, 0.3
    torch.manual_seed(123)
    out = add_dirichlet_noise(p, mask, eps, alpha)
    torch.manual_seed(123)
    again = add_dirichlet_noise(p, mask, eps, alpha)
    assert out.dtype == torch.float32 and torch.equal(out, again)
    assert torch.equal(out[~mask], p[~mask])  # illegal entries untouched
    legal_sum = torch.where(mask, p, torch.zeros_like(p)).sum(1).double()
    got_sum = torch.where(mask, out, torch.zeros_like(out)).sum(1).double()
    rows = mask.any(1)
    assert torch.allclose(got_sum[rows], (1 - eps) * legal_sum[rows] + eps, rtol=0, atol=1e-5)
    assert bool((out[mask] >= 0).all())
    torch.manual_seed(124)
    assert not torch.equal(add_dirichlet_noise(p, mask, eps, alpha), out)


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
@pytest.mark.parametrize("n,trees,sims,R", [(5, 48, 200, 1), (5, 48, 200, 4), (8, 48, 150, 1), (8, 48, 150, 4),
                                            (12, 32, 100, 1), (12, 32, 100, 4), (24, 24, 40, 1), (24, 24, 40, 4)])
def test_device_run_matches_spec(oracle_mod, n, trees, sims, R):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 11 * n + R, trees)
    b = _batch_with_roots(roots, n)
    b.set_stream_base(300)
    m = BatchedMCTS(b, trees, sims, R, 1.25, selection="puct")
    m.begin(0, trees)
    m.run(sims)
    refs = [spec.Search(r, SEED, 300 + t, R, 1.25).run(sims) for t, r in enumerate(roots)]
    _assert_stats_equal(m.root_stats(), refs, n, (n, R))


def _stepwise(m, b, refs, n, trees, sims, root_priors=None, device=False, check_leaves=True):
    """Drives the device search and the specification in lock step with stand-in values and priors; the first
    backup takes root_priors [trees, n*n] when given."""
    import torch
    for k in range(sims):
        status = m.select(trees)
        leaves = b.export_state(trees, trees)
        values = np.zeros((trees, 2), dtype=np.float32)
        priors = np.zeros((trees, n * n), dtype=np.float32)
        for t, ref in enumerate(refs):
            leaf, terminal = ref.select()
            if check_leaves:
                assert np.array_equal(leaves[t], ref.nodes[leaf].state.export_record()), (n, k, t)
                assert status[t] == int(terminal), (n, k, t)
            values[t] = mcts_spec.stand_in_value(leaves[t])
            priors[t] = spec.stand_in_priors(leaves[t], n) if (k > 0 or root_priors is None) else root_priors[t]
            ref.backup(values[t], priors[t])
        if device:
            m.backup(torch.from_numpy(values).cuda(), torch.from_numpy(priors).cuda())
        else:
            m.backup(values, priors)


@pytest.mark.gpu
@pytest.mark.parametrize("n,trees,sims", [(5, 24, 60), (12, 16, 40), (24, 8, 24)])
def test_stepwise_form_matches_spec(oracle_mod, n, trees, sims):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 5 * n, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    m = BatchedMCTS(b, trees, sims, 1, 2.0, selection="puct")
    m.begin(0, trees)
    refs = [spec.Search(r, SEED, t, 1, 2.0) for t, r in enumerate(roots)]
    rng = np.random.default_rng(n)
    root_priors = (rng.random((trees, n * n)) ** 3).astype(np.float32)  # arbitrary, unnormalised
    _stepwise(m, b, refs, n, trees, sims, root_priors)
    _assert_stats_equal(m.root_stats(), refs, n, n)


@pytest.mark.gpu
def test_host_and_device_pointers_give_identical_trees(oracle_mod):
    import torch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 16, 30
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 8, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    out = []
    for device in (False, True):
        m = BatchedMCTS(b, trees, sims, 1, selection="puct")
        m.begin(0, trees)
        refs = [spec.Search(r, SEED, t, 1, 2.0) for t, r in enumerate(roots)]
        _stepwise(m, b, refs, n, trees, sims, device=device)
        out.append(m.root_stats())
        _assert_stats_equal(out[-1], refs, n, device)
        m.close()
    for x, y in zip(*out):
        assert x.tobytes() == y.tobytes()
    # torch tensors on torch's stream, outputs on the device
    b.use_torch_stream()
    m = BatchedMCTS(b, trees, sims, 1, selection="puct")
    m.begin(0, trees)
    status = torch.zeros(trees, dtype=torch.int32, device="cuda")
    refs = [spec.Search(r, SEED, t, 1, 2.0) for t, r in enumerate(roots)]
    for _ in range(sims):
        m.select(trees, status)
        leaves = b.export_state(trees, trees)
        vals = np.stack([mcts_spec.stand_in_value(r) for r in leaves])
        pri = np.stack([spec.stand_in_priors(r, n) for r in leaves])
        for t, ref in enumerate(refs):
            ref.select()
            ref.backup(vals[t], pri[t])
        m.backup(torch.from_numpy(vals).cuda(), torch.from_numpy(pri).cuda())
    dev = (torch.zeros((trees, n * n), dtype=torch.int32, device="cuda"),
           torch.zeros((trees, n * n), dtype=torch.float64, device="cuda"),
           torch.zeros(trees, dtype=torch.int32, device="cuda"))
    m.root_stats(*dev)
    torch.cuda.current_stream().synchronize()
    _assert_stats_equal([x.cpu().numpy() for x in dev], refs, n, "torch")


@pytest.mark.gpu
def test_reproducibility_split_runs_and_sharded_roots(oracle_mod):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n = 8
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 77, 64)
    b = _batch_with_roots(roots, n)
    before = b.export_state()
    m1 = BatchedMCTS(b, 64, 200, 2, selection="puct")
    m1.begin(0, 64)
    m1.run(70)
    m1.run(130)
    split = m1.root_stats()
    m2 = BatchedMCTS(b, 64, 200, 2, selection="puct")
    m2.begin(0, 64)
    m2.run(200)
    whole = m2.root_stats()
    for x, y in zip(split, whole):
        assert x.tobytes() == y.tobytes()
    halves = []
    m3 = BatchedMCTS(b, 32, 200, 2, selection="puct")
    for first in (0, 32):
        m3.begin(first, 32)
        m3.run(200)
        halves.append(m3.root_stats())
    for i in range(3):
        assert np.concatenate([halves[0][i], halves[1][i]]).tobytes() == whole[i].tobytes()
    assert b.export_state().tobytes() == before.tobytes()


@pytest.mark.gpu
def test_launch_counts_and_errors_leave_the_search_exact(oracle_mod):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 16, 40
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 9, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    m = BatchedMCTS(b, trees, sims, 2, selection="puct")
    m.begin(0, trees)
    l0 = b.stats()["kernel_launches"]
    m.run(10)
    assert b.stats()["kernel_launches"] - l0 == 3 * 10
    refs = [spec.Search(r, SEED, t, 2, 2.0).run(10) for t, r in enumerate(roots)]
    _assert_stats_equal(m.root_stats(), refs, n, "run")

    cells = n * n
    vals = np.zeros((trees, 2), dtype=np.float32)
    good = np.full((trees, cells), 1.0 / cells, dtype=np.float32)

    def bad_priors(x):
        p = good.copy()
        p[3, 5] = x
        return p

    uct = BatchedMCTS(b, trees, sims, 2)
    uct.begin(0, trees)
    uct.select(trees)
    with pytest.raises(ValueError, match="UCT"):
        uct.backup(vals, good)
    uct.backup(vals)  # the pending select is still there
    uct.close()

    snap = m.root_stats()
    errors = [lambda: m.backup(vals, good),  # no select pending
              lambda: m.begin(0, trees + 1), lambda: m.run(sims)]
    for call in errors:
        with pytest.raises(ValueError):
            call()
    for x, y in zip(snap, m.root_stats()):
        assert x.tobytes() == y.tobytes()
    for k in range(6):
        l0 = b.stats()["kernel_launches"]
        m.select(trees)
        leaves = b.export_state(trees, trees)
        values = np.stack([mcts_spec.stand_in_value(r) for r in leaves])
        priors = np.stack([spec.stand_in_priors(r, n) for r in leaves])
        for call in (lambda: m.select(trees), lambda: m.run(1),
                     lambda: m._check(m._lib.twixt_mcts_backup_priors(m._h, None, P(priors))),
                     lambda: m.backup(values, bad_priors(float("nan"))),
                     lambda: m.backup(values, bad_priors(-1e-3)),
                     lambda: m.backup(values, bad_priors(float("inf")))):
            with pytest.raises(ValueError):
                call()
        m.backup(values, priors)
        assert b.stats()["kernel_launches"] - l0 == 2
        for t, ref in enumerate(refs):
            leaf, _ = ref.select()
            ref.backup(values[t], priors[t])
    _assert_stats_equal(m.root_stats(), refs, n, "after errors")
    with pytest.raises(MemoryError, match="bytes per tree"):
        BatchedMCTS(b, 1 << 40, 1000, 1, selection="puct")
    with pytest.raises(ValueError):
        BatchedMCTS(b, trees, 40, 2, float("nan"), selection="puct")
    with pytest.raises(ValueError):
        BatchedMCTS(b, trees, 40, 2, selection="alphazero")


@pytest.mark.gpu
def test_self_play_example():
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    try:
        import alphazero_selfplay
    finally:
        sys.path.pop(0)
    from twixt_for_open_spiel_b200 import load_game
    n, games, sims = 8, 64, 16
    trajectories, returns = alphazero_selfplay.self_play(n=n, games=games, sims=sims, temperature=1.0,
                                                         temperature_drop=10, seed=3, verbose=False)
    game = load_game("twixt(board_size=%d)" % n)
    assert len(trajectories) == games and returns.shape == (games, 2)
    for gi, traj in enumerate(trajectories):
        state = game.new_initial_state()
        for step in traj:
            legal = np.zeros(n * n, dtype=bool)
            legal[state.legal_actions()] = True
            assert np.array_equal(step["mask"].astype(bool), legal), gi
            pol = step["policy"]
            assert abs(float(pol.sum()) - 1.0) < 1e-5 and np.all(pol[~legal] == 0), gi
            assert step["player"] == state.current_player(), gi
            assert legal[step["action"]], gi
            state.apply_action(int(step["action"]))
        assert state.is_terminal(), gi
        assert list(returns[gi]) == list(state.returns()), gi


@pytest.mark.gpu
def test_puct_search_at_scale():
    import torch
    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, add_dirichlet_noise
    from twixt_for_open_spiel_b200.producer import ObservationMaskProducer
    n, trees, sims = 12, 8192, 48
    dev = torch.device("cuda:0")
    b = TwixTBatch(n, 2 * trees, 0, SEED)
    b.use_torch_stream()
    group = trees // 8
    for gi in range(8):
        b.playout(gi * group, group, max_plies=3 * gi, want_returns=False, want_lengths=False)
    producer = ObservationMaskProducer(b, max_count=trees)
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(12 * n * (n - 2), n * n + 1)).to(dev)
    m = BatchedMCTS(b, trees, sims, selection="puct")
    m.begin(0, trees)
    player = torch.zeros(trees, dtype=torch.int8, device=dev)
    with torch.no_grad():
        for k in range(sims):
            m.select(trees)
            obs, mask = producer.produce(trees, trees)
            out = net(obs)
            legal = mask.bool()
            pri = torch.softmax(out[:, :n * n].masked_fill(~legal, -1e30), dim=1).float()
            if k == 0:
                pri = add_dirichlet_noise(pri, legal, 0.25, 0.3)
            v = torch.tanh(out[:, n * n])
            b.current_player(trees, trees, out=player)
            v = torch.where(player == 1, -v, v)
            m.backup(torch.stack([v, -v], dim=1).float().contiguous(), pri.contiguous())
    visits, _, best = m.root_stats()
    term = b.is_terminal(0, trees)
    for t in range(trees):
        if term[t]:
            assert visits[t].sum() == 0 and best[t] == -1
        else:
            assert visits[t].sum() == sims - 1 and best[t] >= 0 and visits[t, best[t]] > 0, t
