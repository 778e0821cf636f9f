"""MCTS-Solver searches (twixt_mcts_create_ex with TWIXT_MCTS_SOLVE, twixt_mcts_solver_stats, BatchedMCTS(solve=
True), MCTSBot(solve=True)) against their executable specification tests/solver_spec.py, and proven values against
an exact negamax.  CPU: the specification's own properties, its soundness, and the product's helpers compiled for
the host (tests/solver_harness.cc) running searches node for node against it.  GPU: the device search bit for bit
against the specification (built-in rollouts and the stepwise form), twixt_stats, proofs against negamax, host /
device paths, reproducibility, launch counts, errors, the bot and a search at scale."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import mcts_spec
import puct_spec
import solver_spec as spec

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "twixt_for_open_spiel_b200", "csrc")
SEED = 0x736F6C76
KINDS = ("uct", "puct")


def P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def sh():
    out_dir = os.path.join(HERE, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libsolverharness.so")
    src = os.path.join(HERE, "solver_harness.cc")
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-x", "c++", "-fPIC",
                               "-shared", "-I", CSRC, "-o", so, src])
    lib = C.CDLL(so)
    lib.sh_bytes_per_tree.restype = C.c_int64
    lib.sh_bytes_per_tree.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    lib.sh_proven_value.restype = C.c_int
    lib.sh_proven_value.argtypes = [C.c_int, C.c_int]
    lib.sh_parent_code.restype = C.c_int
    lib.sh_parent_code.argtypes = [C.c_int]
    lib.sh_create.restype = C.c_void_p
    lib.sh_create.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_double, C.c_int, C.c_int]
    lib.sh_destroy.argtypes = [C.c_void_p]
    lib.sh_select.restype = C.c_int
    lib.sh_select.argtypes = [C.c_void_p, C.c_void_p]
    lib.sh_backup.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sh_dump.restype = C.c_int
    lib.sh_dump.argtypes = [C.c_void_p] + [C.c_void_p] * 10
    return lib


def stand_in_priors(n):
    return lambda rec: puct_spec.stand_in_priors(rec, n)


# ------------------------------------------------------------------------------- the specification itself ---
@pytest.mark.parametrize("kind", KINDS)
def test_spec_matches_non_solver_spec_until_the_first_proof(oracle_mod, kind):
    """UCT: identical node for node until the first terminal leaf.  PUCT: until the first non-terminal node is
    proven (PUCT already scores terminal children by their outcome)."""
    n = 5
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 21, 12)
    checked = 0
    for i, root in enumerate(roots):
        if root.is_terminal():
            continue
        base = (puct_spec.Search if kind == "puct" else mcts_spec.Search)(root, SEED, 40 + i, 1, 1.5)
        sol = spec.make(kind, root, SEED, 40 + i, 1, 1.5)
        for k in range(300):
            leaf, status = sol.select()
            bleaf, bterm = base.select()
            assert (leaf, status) == (bleaf, int(bterm)), (i, k)
            v = sol.rollout_value(leaf) if status == 0 else None
            sol.backup(v)
            base.backup(v)
            if kind == "uct":
                assert [(x.n, x.edge_n, x.edge_w) for x in sol.nodes] == [(x.n, x.edge_n, x.edge_w) for x in base.nodes]
                if status == spec.LEAF_TERMINAL:
                    break
            else:
                assert [d[:7] for d in sol.dump()] == [tuple(d) for d in base.dump()], (i, k)
                if any(nd.outcome is not None and not nd.state.is_terminal() for nd in sol.nodes):
                    break
        checked += 1
    assert checked >= 8


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


@pytest.mark.parametrize("n", [5, 8])
def test_spec_uct_proves_a_win_in_one_and_stops(oracle_mod, n):
    g = oracle_mod.OracleGame(n)
    root, win = winning_root(g, n)
    L = len(root.legal_actions())
    s = spec.UctSolveSearch(root, SEED, 3, 1)
    for k in range(L + 1):
        s.simulate()
        if s.finished:
            break
    assert s.finished, "not proven within L + 1 simulations"
    proven, ret, values, sims = s.solver_stats(n)
    mover = root.current_player()
    assert proven == 1 and ret[mover] == 1.0 and ret[1 - mover] == -1.0
    best = s.root_stats(n)[2]
    end = root.clone()
    end.apply_action(best)
    assert end.returns()[mover] == 1.0 and values[best] == 1  # the first winning move reached, maybe not `win`
    s.run(20)
    assert s.solver_stats(n)[3] == sims and s.k == sims + 20


@pytest.mark.parametrize("kind", KINDS)
def test_spec_terminal_root_is_proven_at_simulation_zero(oracle_mod, kind):
    n = 6
    g = oracle_mod.OracleGame(n)
    term = g.new_initial_state()
    for a in term.clone().playout_philox(SEED, 5):
        term.apply_action(a)
    s = spec.make(kind, term, SEED, 4)
    assert not s.finished
    s.simulate()
    assert s.finished
    proven, ret, values, sims = s.solver_stats(n)
    assert proven == 1 and list(ret) == list(term.returns()) and sims == 1 and (values == spec.UNPROVEN).all()
    assert s.select() == (None, spec.LEAF_SOLVED)


def test_spec_proofs_agree_with_negamax(oracle_mod):
    """Independent of the specification's proof rule: every proven root value and root edge value equals the
    exact game value, and wins, losses and draws all occur among them."""
    n = 5
    g = oracle_mod.OracleGame(n)
    memo = {}
    seen = set()
    proven_roots = 0
    for kind in KINDS:
        for i, root in enumerate(spec.near_end_roots(g, n, 5 + len(kind), 60, back=(2, 3, 4, 5, 6))):
            if len(root.legal_actions()) > 11:
                continue
            s = spec.make(kind, root, SEED, 100 + i, 1, 1.0)
            s.run(300)
            proven, ret, values, _ = s.solver_stats(n)
            ply = int(root.export_record()[0])
            if proven:
                proven_roots += 1
                v = spec.negamax(root, memo)
                assert int(ret[ply & 1]) == v and int(ret[1 - (ply & 1)]) == -v, (kind, i)
                seen.add(v)
            for a in np.flatnonzero(values != spec.UNPROVEN):
                ch = root.clone()
                ch.apply_action(int(a))
                assert int(values[a]) == -spec.negamax(ch, memo), (kind, i, a)
                seen.add(int(values[a]))
    assert proven_roots >= 20 and seen == {-1, 0, 1}


# ----------------------------------------------------------------------- host harness vs specification ---
def harness_search(sh, kind, root, n, seed, T, R, c, sims, value_fn=None, prior_fn=None):
    rec = np.ascontiguousarray(root.export_record())
    h = sh.sh_create(P(rec), n, seed, T, R, c, sims, int(kind == "puct"))
    leaf = np.zeros_like(rec)
    statuses = []
    try:
        for _ in range(sims):
            status = sh.sh_select(h, P(leaf))
            statuses.append(status)
            vals = pri = None
            if status == 0 and value_fn is not None:
                vals = np.ascontiguousarray(value_fn(leaf), dtype=np.float32)
            if status == 0 and prior_fn is not None:
                pri = np.ascontiguousarray(prior_fn(leaf), dtype=np.float32)
            sh.sh_backup(h, None if vals is None else P(vals), None if pri is None else P(pri))
        S, M = sims + 1, n * (n - 2)
        parent, action, legal = (np.zeros(S, dtype=np.int32) for _ in range(3))
        visits = np.zeros(S, dtype=np.uint32)
        en = np.zeros((S, M), dtype=np.uint32)
        ew = np.zeros((S, M), dtype=np.float64)
        ep = np.zeros((S, M), dtype=np.float32)
        eo = np.zeros((S, M), dtype=np.uint8)
        root_code = np.zeros(1, dtype=np.int32)
        best = np.zeros(1, dtype=np.int32)
        count = sh.sh_dump(h, P(parent), P(action), P(visits), P(legal), P(en), P(ew), P(ep), P(eo), P(root_code),
                           P(best))
    finally:
        sh.sh_destroy(h)
    return count, parent, action, visits, legal, en, ew, ep, eo, int(root_code[0]), int(best[0]), statuses


def spec_search(kind, root, T, R, c, sims, value_fn=None, prior_fn=None):
    s = spec.make(kind, root, SEED, T, R, c)
    statuses = []
    for _ in range(sims):
        leaf, status = s.select()
        statuses.append(status)
        if status != 0:
            s.backup(None) if kind == "uct" else s.backup(None, None)
            continue
        rec = s.nodes[leaf].state.export_record()
        v = s.rollout_value(leaf) if value_fn is None else value_fn(rec)
        if kind == "uct":
            s.backup(v)
        else:
            s.backup(v, None if prior_fn is None else prior_fn(rec))
    return s, statuses


def assert_harness_matches(got, ref, ref_statuses, n, tag):
    count, parent, action, visits, legal, en, ew, ep, eo, root_code, best, statuses = got
    assert statuses == ref_statuses, tag
    dump = ref.dump()
    assert count == len(dump), tag
    for k, (par, act, nn, L, e_n, e_w, e_p, codes) in enumerate(dump):
        assert (parent[k], action[k], visits[k], legal[k]) == (par, act, nn, L), (tag, k)
        if L > 0:
            assert en[k, :L].tolist() == list(e_n), (tag, k)
            assert ew[k, :L].tobytes() == np.asarray(e_w, dtype=np.float64).tobytes(), (tag, k)
            if e_p is not None:
                assert ep[k, :L].tobytes() == np.asarray(e_p, dtype=np.float32).tobytes(), (tag, k)
            assert eo[k, :L].tolist() == codes, (tag, k)
    assert root_code == ref.root_code(), tag
    assert best == ref.root_stats(n)[2], tag


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [5, 8, 12])
def test_harness_matches_spec_node_for_node(sh, oracle_mod, kind, n):
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 60 + n, 6) + spec.near_end_roots(g, n, 61 + n, 4)
    sims_for = {5: 150, 8: 100, 12: 50}
    finished = 0
    for i, root in enumerate(roots):
        R = 1 if i % 2 == 0 else 4
        c = 2.0 if i % 2 == 0 else 0.7
        T = 1000 * n + i
        sims = sims_for[n]
        ref, st = spec_search(kind, root, T, R, c, sims)
        assert_harness_matches(harness_search(sh, kind, root, n, SEED, T, R, c, sims), ref, st, n, (n, i, "rollouts"))
        finished += ref.finished
        pri = stand_in_priors(n) if kind == "puct" else None
        ref, st = spec_search(kind, root, T, 1, c, sims, mcts_spec.stand_in_value, pri)
        got = harness_search(sh, kind, root, n, SEED, T, 1, c, sims, mcts_spec.stand_in_value, pri)
        assert_harness_matches(got, ref, st, n, (n, i, "stand-in"))
        finished += ref.finished
    assert finished >= 2  # terminal roots at least


def test_byte_formula_and_proof_helpers(sh):
    # n = 12: rw = 112 words; UCT + solve: 401 * (448 + 8 + 19 * 120) + 17 + 8 * 142 + 4 * (448 + 16)
    assert sh.sh_bytes_per_tree(12, 400, 4, 0) == 401 * (448 + 8 + 19 * 120) + 17 + 8 * 142 + 4 * (448 + 16)
    assert sh.sh_bytes_per_tree(12, 400, 4, 1) == 401 * (448 + 8 + 27 * 120) + 17 + 8 * 142 + 4 * (448 + 16)
    for mx in range(4):
        for all_proven in (0, 1):
            v = sh.sh_proven_value(mx, all_proven)
            assert v == (mx - 2 if (mx == 3 or all_proven) else spec.UNPROVEN)
    assert [sh.sh_parent_code(v) for v in (-1, 0, 1)] == [3, 2, 1]


# ---------------------------------------------------------------------------------------------- GPU ---
def _batch_with_roots(roots, n, seed=SEED, extra=0):
    from twixt_for_open_spiel_b200 import TwixTBatch
    b = TwixTBatch(n, len(roots) + extra, 0, seed)
    b.import_state(np.stack([r.export_record() for r in roots]), 0)
    return b


def _assert_stats_equal(m, refs, n, tag):
    visits, sums, best = m.root_stats()
    proven, ret, values, sims = m.solver_stats()
    for t, ref in enumerate(refs):
        v, w, bst = ref.root_stats(n)
        assert np.array_equal(visits[t], v), (tag, t)
        assert sums[t].tobytes() == w.tobytes(), (tag, t)
        assert best[t] == bst, (tag, t)
        rp, rr, rv, rs = ref.solver_stats(n)
        assert (proven[t], sims[t]) == (rp, rs), (tag, t)
        assert ret[t].tobytes() == rr.tobytes(), (tag, t)
        assert np.array_equal(values[t], rv), (tag, t)


class _Counted:
    """Counts the plies and games of a specification's rollouts (what twixt_stats must add)."""

    def __init__(self):
        self.plies = 0
        self.games = 0

    def wrap(self, s):
        orig = s.rollout_value

        def rollout_value(leaf):
            for r in range(s.R):
                st = s.nodes[leaf].state.clone()
                self.plies += len(st.playout_philox(s.seed, mcts_spec.rollout_stream(s.T, s.k, s.R, r)))
                self.games += 1
            return orig(leaf)
        s.rollout_value = rollout_value
        return s


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,trees,sims", [(5, 48, 200), (8, 48, 150), (12, 30, 100), (24, 18, 40)])
@pytest.mark.parametrize("R", [1, 4])
def test_device_run_matches_spec(oracle_mod, kind, n, trees, sims, R):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 13 * n + R, trees - 6) + spec.near_end_roots(g, n, n + R, 6)
    b = _batch_with_roots(roots, n)
    b.set_stream_base(500)
    m = BatchedMCTS(b, trees, sims, R, 1.25, selection=kind, solve=True)
    m.begin(0, trees)
    b.stats_reset()
    m.run(sims)
    counter = _Counted()
    refs = [counter.wrap(spec.make(kind, r, SEED, 500 + t, R, 1.25)).run(sims) for t, r in enumerate(roots)]
    _assert_stats_equal(m, refs, n, (kind, n, R))
    st = b.stats()
    assert (st["plies"], st["games"]) == (counter.plies, counter.games), (kind, n, R)
    assert sum(r.finished for r in refs) >= 4


def _stepwise(m, b, refs, kind, n, trees, sims, device=False, poison=True):
    """Drives the device search and the specification in lock step with stand-in values and priors; rows of
    finished trees are poisoned with NaN (device tensors)."""
    import torch
    seen_solved = 0
    for k in range(sims):
        before = b.export_state(trees, trees)
        status = m.select(trees)
        leaves = b.export_state(trees, trees)
        values = np.zeros((trees, 2), dtype=np.float32)
        priors = np.zeros((trees, n * n), dtype=np.float32)
        for t, ref in enumerate(refs):
            leaf, st = ref.select()
            assert status[t] == st, (n, k, t)
            if st == spec.LEAF_SOLVED:
                seen_solved += 1
                assert leaves[t].tobytes() == before[t].tobytes(), (n, k, t)
                values[t] = np.nan
                priors[t] = np.nan
                ref.backup(None) if kind == "uct" else ref.backup(None, None)
                continue
            assert np.array_equal(leaves[t], ref.nodes[leaf].state.export_record()), (n, k, t)
            values[t] = mcts_spec.stand_in_value(leaves[t])
            priors[t] = puct_spec.stand_in_priors(leaves[t], n)
            ref.backup(values[t]) if kind == "uct" else ref.backup(values[t], priors[t])
        if device or poison:
            m.backup(torch.from_numpy(values).cuda(), torch.from_numpy(priors).cuda() if kind == "puct" else None)
        else:
            m.backup(values, priors if kind == "puct" else None)
    return seen_solved


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,trees,sims", [(5, 24, 80), (8, 24, 60), (12, 12, 30)])
def test_stepwise_form_matches_spec(oracle_mod, kind, n, trees, sims):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 7 * n, trees // 2) + spec.near_end_roots(g, n, 8 * n, trees - trees // 2)
    b = _batch_with_roots(roots, n, extra=trees)
    m = BatchedMCTS(b, trees, sims, 1, 2.0, selection=kind, solve=True)
    m.begin(0, trees)
    refs = [spec.make(kind, r, SEED, t, 1, 2.0) for t, r in enumerate(roots)]
    assert _stepwise(m, b, refs, kind, n, trees, sims) > 0
    _assert_stats_equal(m, refs, n, (kind, n))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_twixt_stats_after_stepwise_finish_then_run(oracle_mod, kind):
    """Trees that finish during stepwise calls, then `run`: their never-written rollout slots add nothing."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees = 8, 32
    g = oracle_mod.OracleGame(n)
    roots = spec.near_end_roots(g, n, 31, trees, back=(1, 2, 3))
    b = _batch_with_roots(roots, n, extra=trees)
    m = BatchedMCTS(b, trees, 120, 2, 2.0, selection=kind, solve=True)
    m.begin(0, trees)
    refs = [spec.make(kind, r, SEED, t, 2, 2.0) for t, r in enumerate(roots)]
    _stepwise(m, b, refs, kind, n, trees, 40)
    assert sum(r.finished for r in refs) >= trees // 4
    b.stats_reset()
    m.run(80)
    counter = _Counted()
    for ref in refs:
        counter.wrap(ref).run(80)
    st = b.stats()
    assert (st["plies"], st["games"]) == (counter.plies, counter.games)
    _assert_stats_equal(m, refs, n, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_device_proofs_agree_with_negamax(oracle_mod, kind):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees = 5, 3000
    g = oracle_mod.OracleGame(n)
    roots = spec.near_end_roots(g, n, 17 + len(kind), trees, back=(2, 3, 4, 5, 6))
    b = _batch_with_roots(roots, n)
    m = BatchedMCTS(b, trees, 400, 1, 1.0, selection=kind, solve=True)
    m.begin(0, trees)
    m.run(400)
    proven, ret, values, _ = m.solver_stats()
    memo = {}
    seen = set()
    checked = 0
    for t, root in enumerate(roots):
        if len(root.legal_actions()) > 8:  # negamax in Python stays within seconds up to here
            continue
        checked += 1
        ply = int(root.export_record()[0])
        if proven[t]:
            v = spec.negamax(root, memo)
            assert (int(ret[t, ply & 1]), int(ret[t, 1 - (ply & 1)])) == (v, -v), t
            seen.add(v)
        for a in np.flatnonzero(values[t] != spec.UNPROVEN):
            ch = root.clone()
            ch.apply_action(int(a))
            assert int(values[t, a]) == -spec.negamax(ch, memo), (t, a)
    assert checked > trees // 2 and proven.sum() > trees // 2 and seen == {-1, 0, 1}


@pytest.mark.gpu
def test_host_and_device_pointers_split_runs_and_shards(oracle_mod):
    import torch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 32, 100
    g = oracle_mod.OracleGame(n)
    roots = spec.near_end_roots(g, n, 41, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    before = b.export_state()
    for kind in KINDS:
        whole = BatchedMCTS(b, trees, sims, 2, selection=kind, solve=True)
        whole.begin(0, trees)
        whole.run(sims)
        host = whole.solver_stats() + whole.root_stats()
        dev = (torch.zeros(trees, dtype=torch.uint8, device="cuda"),
               torch.zeros((trees, 2), dtype=torch.float32, device="cuda"),
               torch.zeros((trees, n * n), dtype=torch.int8, device="cuda"),
               torch.zeros(trees, dtype=torch.int32, device="cuda"))
        whole.solver_stats(*dev)
        torch.cuda.synchronize()
        for x, y in zip(host[:4], dev):
            assert x.tobytes() == y.cpu().numpy().tobytes(), kind
        split = BatchedMCTS(b, trees, sims, 2, selection=kind, solve=True)
        split.begin(0, trees)
        split.run(30)
        split.run(70)
        for x, y in zip(host, split.solver_stats() + split.root_stats()):
            assert x.tobytes() == y.tobytes(), kind
        half = BatchedMCTS(b, trees // 2, sims, 2, selection=kind, solve=True)
        parts = []
        for first in (0, trees // 2):
            half.begin(first, trees // 2)
            half.run(sims)
            parts.append(half.solver_stats() + half.root_stats())
        for i in range(7):
            assert np.concatenate([parts[0][i], parts[1][i]]).tobytes() == host[i].tobytes(), (kind, i)
        for mm in (whole, split, half):
            mm.close()
    assert b.export_state().tobytes() == before.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_launch_counts_and_errors_leave_the_trees_exact(oracle_mod, kind):
    from twixt_for_open_spiel_b200 import _lib
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 16, 60
    g = oracle_mod.OracleGame(n)
    roots = spec.near_end_roots(g, n, 51, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    counts = []
    for solve in (False, True):
        m = BatchedMCTS(b, trees, sims, 2, selection=kind, solve=solve)
        m.begin(0, trees)
        l0 = b.stats()["kernel_launches"]
        m.run(10)
        m.select(trees)
        m.backup(np.zeros((trees, 2), dtype=np.float32))
        m.root_stats()
        counts.append(b.stats()["kernel_launches"] - l0)
        if not solve:
            with pytest.raises(ValueError, match="TWIXT_MCTS_SOLVE"):
                m.solver_stats()
            m.close()
    assert counts[0] == counts[1] == 3 * 10 + 2 + 1
    l0 = b.stats()["kernel_launches"]
    m.solver_stats()
    assert b.stats()["kernel_launches"] - l0 == 1
    refs = [spec.make(kind, r, SEED, t, 2, 2.0) for t, r in enumerate(roots)]
    for ref in refs:
        ref.run(10)
        leaf, st = ref.select()
        z = np.zeros(2, dtype=np.float32)
        ref.backup(None if st else z) if kind == "uct" else ref.backup(None if st else z, None)
    _assert_stats_equal(m, refs, n, "before errors")
    m.select(trees)
    with pytest.raises(ValueError):
        m.solver_stats()  # a select awaits its backup
    m.backup(np.zeros((trees, 2), dtype=np.float32))
    for ref in refs:
        leaf, st = ref.select()
        z = np.zeros(2, dtype=np.float32)
        ref.backup(None if st else z) if kind == "uct" else ref.backup(None if st else z, None)
    _assert_stats_equal(m, refs, n, "after errors")
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.twixt_mcts_create_ex(b._h, trees, sims, 2, 2.0, 4, C.byref(h)) == _lib.EINVAL and not h.value
    assert lib.twixt_mcts_create_ex(b._h, trees, sims, 2, 2.0, 0x80000003, C.byref(h)) == _lib.EINVAL
    fresh = BatchedMCTS(b, trees, sims, 2, selection=kind, solve=True)
    with pytest.raises(ValueError, match="no search begun"):
        fresh.solver_stats()
    fresh.close()
    _assert_stats_equal(m, refs, n, "after create errors")


@pytest.mark.gpu
def test_flags_zero_and_puct_are_the_old_constructors(oracle_mod):
    from twixt_for_open_spiel_b200 import _lib
    n, trees, sims = 8, 16, 40
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 3, trees)
    b = _batch_with_roots(roots, n)
    lib = _lib.load()
    cells = n * n
    for flags, old in ((0, lib.twixt_mcts_create), (1, lib.twixt_mcts_create_puct)):
        outs = []
        for make in (lambda h: lib.twixt_mcts_create_ex(b._h, trees, sims, 2, 1.5, flags, C.byref(h)),
                     lambda h: old(b._h, trees, sims, 2, 1.5, C.byref(h))):
            h = C.c_void_p()
            assert make(h) == 0
            assert lib.twixt_mcts_begin(h, 0, trees) == 0 and lib.twixt_mcts_run(h, sims) == 0
            v = np.zeros((trees, cells), dtype=np.int32)
            w = np.zeros((trees, cells), dtype=np.float64)
            best = np.zeros(trees, dtype=np.int32)
            assert lib.twixt_mcts_root_stats(h, P(v), P(w), P(best)) == 0
            assert lib.twixt_mcts_solver_stats(h, None, None, None, None) == _lib.EINVAL
            lib.twixt_mcts_destroy(h)
            outs.append(v.tobytes() + w.tobytes() + best.tobytes())
        assert outs[0] == outs[1], flags


def winning_positions(g, count):
    """[(history, state)] of positions whose player to move wins with one of its legal actions."""
    out = []
    for s in range(5000):
        st = g.new_initial_state()
        acts = st.clone().playout_philox(SEED, s)
        for a in acts[:-1]:
            st.apply_action(a)
        end = st.clone()
        end.apply_action(acts[-1])
        if end.returns()[st.current_player()] == 1.0:
            out.append((acts[:-1], st))
            if len(out) == count:
                return out
    raise AssertionError("not enough positions one move from a win")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [6, 8])
def test_bot_with_solver_plays_a_winning_move(oracle_mod, n):
    from twixt_for_open_spiel_b200 import load_game
    from twixt_for_open_spiel_b200.mcts import MCTSBot
    g = oracle_mod.OracleGame(n)
    game = load_game("twixt(board_size=%d)" % n)
    bot = MCTSBot(game, max_simulations=400, n_rollouts=1, seed=3, solve=True)
    for i, (history, root) in enumerate(winning_positions(g, 6)):
        state = game.new_initial_state()
        for a in history:
            state.apply_action(a)
        act = bot.step(state)
        end = root.clone()
        end.apply_action(act)
        assert end.is_terminal() and end.returns()[root.current_player()] == 1.0, i
    bot.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_solver_at_scale(oracle_mod, kind):
    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims, R = 8, 8192, 200, 2
    g = oracle_mod.OracleGame(n)
    rng = random.Random(9)
    sample = sorted(rng.sample(range(trees), 24))
    roots = spec.near_end_roots(g, n, 77, trees, back=(3, 4, 5, 6, 8))
    b = TwixTBatch(n, trees, 0, SEED)
    b.import_state(np.stack([r.export_record() for r in roots]), 0)
    m = BatchedMCTS(b, trees, sims, R, selection=kind, solve=True)
    m.begin(0, trees)
    m.run(sims)
    proven, ret, values, simulations = m.solver_stats()
    visits, sums, best = m.root_stats()
    for t in sample:
        ref = spec.make(kind, roots[t], SEED, t, R, 2.0).run(sims)
        v, w, bst = ref.root_stats(n)
        rp, rr, rv, rs = ref.solver_stats(n)
        assert np.array_equal(visits[t], v) and sums[t].tobytes() == w.tobytes() and best[t] == bst, t
        assert (proven[t], simulations[t]) == (rp, rs) and ret[t].tobytes() == rr.tobytes(), t
        assert np.array_equal(values[t], rv), t
    # many of these endgames get proven (PUCT with uniform priors proves fewer than UCT in 200 simulations), and
    # most proven trees stopped early
    assert proven.mean() > 0.3 and (simulations[proven == 1] < sims).mean() > 0.5
