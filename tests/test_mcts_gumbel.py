"""Gumbel AlphaZero search (twixt_mcts_create_gumbel, BatchedMCTS(selection="gumbel")) against its executable
specification tests/gumbel_spec.py.  CPU: mcts_exp and the considered-visits table bit for bit, a hand-computed
node, the specification's own properties, and the product's helpers compiled for the host (tests/gumbel_harness.cc)
running searches node for node against it.  GPU: the device search bit for bit against the specification (run and
the stepwise form, zero and non-zero noise, host and device pointers), split runs, determinism, errors, the budget,
launch counts, the self-play example and a search at scale."""
import ctypes as C
import math
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import gumbel_spec as spec
import mcts_spec

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "twixt_for_open_spiel_b200", "csrc")
SEED = 0x67756D62


def P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def gh():
    out_dir = os.path.join(HERE, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libgumbelharness.so")
    src = os.path.join(HERE, "gumbel_harness.cc")
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-x", "c++", "-fPIC",
                               "-shared", "-I", CSRC, "-o", so, src])
    lib = C.CDLL(so)
    lib.gh_exp.restype = C.c_double
    lib.gh_exp.argtypes = [C.c_double]
    lib.gh_considered_visits.argtypes = [C.c_int, C.c_int, C.c_void_p]
    lib.gh_bytes_per_tree.restype = C.c_int64
    lib.gh_bytes_per_tree.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.gh_create.restype = C.c_void_p
    lib.gh_create.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_double,
                              C.c_double, C.c_void_p]
    lib.gh_destroy.argtypes = [C.c_void_p]
    lib.gh_select.restype = C.c_int
    lib.gh_select.argtypes = [C.c_void_p, C.c_void_p]
    lib.gh_backup.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gh_dump.restype = C.c_int
    lib.gh_dump.argtypes = [C.c_void_p] + [C.c_void_p] * 8
    lib.gh_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


def mctx_sequence(max_num_considered_actions, num_simulations):
    """A literal transcription of mctx seq_halving.get_sequence_of_considered_visits."""
    if max_num_considered_actions <= 1:
        return tuple(range(num_simulations))
    log2max = int(math.ceil(math.log2(max_num_considered_actions)))
    sequence = []
    visits = [0] * max_num_considered_actions
    num_considered = max_num_considered_actions
    while len(sequence) < num_simulations:
        num_extra_visits = max(1, int(num_simulations / (log2max * num_considered)))
        for _ in range(num_extra_visits):
            sequence.extend(visits[:num_considered])
            for i in range(num_considered):
                visits[i] += 1
        num_considered = max(2, num_considered // 2)
    return tuple(sequence[:num_simulations])


def noise_for(n, count, seed):
    rng = np.random.default_rng(seed)
    u = rng.random((count, n * n)).clip(1e-300, None)
    return (-np.log(-np.log(u))).astype(np.float32)


def stand_in_value(record):
    return mcts_spec.stand_in_value(record)


# ------------------------------------------------------------------------------------------- arithmetic ---
def test_mcts_exp_is_bit_exact_and_within_two_ulp(gh):
    rng = random.Random(7)
    pts = [rng.uniform(-746.0, 0.0) for _ in range(100000)] + [rng.uniform(-2.0, 0.0) for _ in range(20000)]
    pts += [0.0, -0.0, -1e-300, -746.0, -745.5, -745.1, -744.4, -708.4, -708.3, -0.5 * math.log(2), -math.log(2)]
    for x in pts:
        got = gh.gh_exp(x)
        ref = spec.mcts_exp(x)
        assert got.hex() == ref.hex(), x
        exact = math.exp(x)
        assert abs(got - exact) <= 2 * math.ulp(exact), x
    assert spec.mcts_exp(-746.5) == 0.0 and gh.gh_exp(-1e9) == 0.0 and spec.mcts_exp(0.0) == 1.0


def test_considered_visits_table_matches_mctx(gh):
    for budget in (0, 1, 2, 3, 7, 15, 16, 63, 199, 399, 1000):
        for m in range(0, 33):
            ref = list(mctx_sequence(m, budget))
            assert spec.considered_visits(m, budget) == ref, (m, budget)
            out = np.zeros(max(budget, 1), dtype=np.int32)
            gh.gh_considered_visits(m, budget, P(out))
            assert out[:budget].tolist() == ref, (m, budget)
    assert spec.considered_table(4, 10) == [list(mctx_sequence(m, 10)) for m in range(5)]


def test_hand_computed_node():
    """pi, v_mix, q^, sigma and pi' of one node against a plain float64 restatement of mctx."""
    logits = [0.5, -1.25, 2.0, 0.0, -30.0, 1.5, 3.25]
    visits = [3, 0, 5, 1, 0, 0, 2]
    sums = [1.5, 0.0, -2.0, 0.75, 0.0, 0.0, 1.0]
    raw, c_visit, c_scale = -0.3, 50.0, 0.1
    cq = spec.completed_q(logits, visits, sums, raw, c_visit, c_scale)
    l = np.asarray(logits)
    n = np.asarray(visits, dtype=np.float64)
    w = np.asarray(sums)
    pi = np.maximum(np.exp(l - l.max()) / np.exp(l - l.max()).sum(), np.finfo(np.float64).tiny)
    q = np.where(n > 0, w / np.where(n > 0, n, 1), 0.0)
    sp = pi[n > 0].sum()
    v_mix = (raw + n.sum() * (pi[n > 0] * q[n > 0] / sp).sum()) / (n.sum() + 1)
    qc = np.where(n > 0, q, v_mix)
    qh = (qc - qc.min()) / max(qc.max() - qc.min(), 1e-8)
    sigma = (c_visit + n.max()) * c_scale * qh
    x = l + sigma
    pi2 = np.exp(x - x.max()) / np.exp(x - x.max()).sum()
    assert abs(cq["v_mix"] - v_mix) < 1e-12
    assert np.allclose(cq["pi"], pi, rtol=0, atol=1e-12)
    assert np.allclose(cq["q"], qc, rtol=0, atol=1e-12)
    assert np.allclose(cq["sigma"], sigma, rtol=0, atol=1e-12)
    assert np.allclose(spec.improved_policy(logits, cq["sigma"]), pi2, rtol=0, atol=1e-12)
    interior = pi2 - n / (1 + n.sum())
    assert spec.argmax(list(pi2 - n / (1 + n.sum()))) == int(np.argmax(interior))
    # no visited edge: v_mix is the raw value and sigma is 0
    cq0 = spec.completed_q(logits, [0] * 7, [0.0] * 7, raw, c_visit, c_scale)
    assert cq0["v_mix"] == raw and cq0["sigma"] == [0.0] * 7


# ---------------------------------------------------------------------------------- the specification ---
def test_spec_sequential_halving_visits_follow_the_table(oracle_mod):
    n, sims, mc = 8, 64, 8
    g = oracle_mod.OracleGame(n)
    root = g.new_initial_state()
    root.apply_action(20)
    s = spec.Search(root, SEED, 3, max_simulations=sims, max_considered=mc, gumbel=noise_for(n, 1, 1)[0])
    logit_fn = lambda rec: spec.stand_in_logits(rec, n)  # noqa: E731
    seen = set()
    for i in range(sims):
        r = s.nodes[0]
        before = {c.action: c.explore_count for c in r.children}
        s.simulate(stand_in_value, logit_fn)
        if i == 0:
            continue
        after = {c.action: c.explore_count for c in r.children}
        moved = [a for a in after if after[a] != before[a]]
        assert len(moved) == 1
        m = min(mc, len(r.children))
        assert before[moved[0]] == s.table[m][i - 1], i
        seen.add(moved[0])
    assert len(seen) == mc
    visits = sorted((c.explore_count for c in s.nodes[0].children), reverse=True)
    assert sum(visits) == sims - 1
    a, pol = s.gumbel_stats(n)
    assert a >= 0 and abs(float(pol.sum(dtype=np.float64)) - 1.0) < 1e-5
    assert s.nodes[0].edges()[[c.action for c in s.nodes[0].edges()].index(a)].explore_count == visits[0]


def test_spec_zero_noise_uniform_logits_takes_the_lowest_edges_first(oracle_mod):
    n, sims, mc = 6, 40, 4
    g = oracle_mod.OracleGame(n)
    root = g.new_initial_state()
    s = spec.Search(root, SEED, 5, max_simulations=sims, max_considered=mc).run(sims)
    legal = root.legal_actions()
    assert [s.nodes[k].action for k in range(1, mc + 1)] == legal[:mc]
    assert all(s.nodes[k].parent_slot == 0 for k in range(1, mc + 1))
    v, _, _ = s.root_stats(n)
    assert set(np.nonzero(v)[0].tolist()) == set(legal[:mc])


def test_spec_one_considered_move_and_more_than_legal(oracle_mod):
    n, sims = 5, 30
    g = oracle_mod.OracleGame(n)
    root = g.new_initial_state()
    noise = noise_for(n, 1, 9)[0]
    logit_fn = lambda rec: spec.stand_in_logits(rec, n)  # noqa: E731
    s1 = spec.Search(root, SEED, 1, max_simulations=sims, max_considered=1, gumbel=noise).run(sims, stand_in_value,
                                                                                              logit_fn)
    v, _, best = s1.root_stats(n)
    legal = root.legal_actions()
    l0 = spec.stand_in_logits(root.export_record(), n)
    top = max(legal, key=lambda a: (float(noise[a]) + float(l0[a]), -a))
    assert v.sum() == sims - 1 and v[top] == sims - 1 and best == top
    L = len(legal)
    big = spec.Search(root, SEED, 1, max_simulations=sims, max_considered=1000, gumbel=noise).run(
        sims, stand_in_value, logit_fn)
    exact = spec.Search(root, SEED, 1, max_simulations=sims, max_considered=L, gumbel=noise).run(
        sims, stand_in_value, logit_fn)
    assert repr(big.dump()) == repr(exact.dump())


def test_spec_terminal_root(oracle_mod):
    g = oracle_mod.OracleGame(6)
    term = g.new_initial_state()
    for a in term.clone().playout_philox(SEED, 5):
        term.apply_action(a)
    s = spec.Search(term, SEED, 4, max_simulations=10).run(10)
    a, pol = s.gumbel_stats(6)
    assert a == -1 and not pol.any() and s.nodes[0].explore_count == 10 and len(s.nodes) == 1


# ------------------------------------------------------------------------ host harness vs specification ---
def harness_search(gh, root, n, T, R, sims, mc, noise, value_fn=None, logit_fn=None, c_visit=50.0, c_scale=0.1):
    rec = np.ascontiguousarray(root.export_record())
    h = gh.gh_create(P(rec), n, SEED, T, R, sims, mc, c_visit, c_scale, None if noise is None else P(noise))
    leaf = np.zeros_like(rec)
    try:
        for _ in range(sims):
            terminal = gh.gh_select(h, P(leaf))
            vals = lg = None
            if not terminal and value_fn is not None:
                vals = np.ascontiguousarray(value_fn(leaf), dtype=np.float32)
            if not terminal and logit_fn is not None:
                lg = np.ascontiguousarray(logit_fn(leaf), dtype=np.float32)
            gh.gh_backup(h, None if vals is None else P(vals), None if lg is None else P(lg))
        S, M = sims + 1, n * (n - 2)
        parent, action, legal = (np.zeros(S, dtype=np.int32) for _ in range(3))
        visits = np.zeros(S, dtype=np.uint32)
        value = np.zeros(S, dtype=np.float64)
        en = np.zeros((S, M), dtype=np.uint32)
        ew = np.zeros((S, M), dtype=np.float64)
        el = np.zeros((S, M), dtype=np.float32)
        count = gh.gh_dump(h, P(parent), P(action), P(visits), P(legal), P(value), P(en), P(ew), P(el))
        act = np.zeros(1, dtype=np.int32)
        pol = np.zeros(n * n, dtype=np.float32)
        gh.gh_stats(h, P(act), P(pol))
    finally:
        gh.gh_destroy(h)
    return count, parent, action, visits, legal, value, en, ew, el, int(act[0]), pol


def assert_harness_matches(got, ref, n, tag):
    count, parent, action, visits, legal, value, en, ew, el, act, pol = got
    dump = ref.dump()
    assert count == len(dump), tag
    for k, (par, a, nn, L, e_n, e_w, e_l, v) in enumerate(dump):
        assert (parent[k], action[k], visits[k], legal[k]) == (par, a, nn, L), (tag, k)
        assert value[k].hex() == float(v).hex(), (tag, k)
        if L > 0:
            assert en[k, :L].tolist() == e_n, (tag, k)
            assert ew[k, :L].tobytes() == np.asarray(e_w, dtype=np.float64).tobytes(), (tag, k)
            assert el[k, :L].tobytes() == np.asarray(e_l, dtype=np.float32).tobytes(), (tag, k)
    ra, rp = ref.gumbel_stats(n)
    assert act == ra and pol.tobytes() == rp.tobytes(), tag


@pytest.mark.parametrize("n", [5, 8, 12])
def test_harness_matches_spec_node_for_node(gh, oracle_mod, n):
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 70 + n, 6)
    sims_for = {5: 120, 8: 80, 12: 40}
    logit_fn = lambda rec: spec.stand_in_logits(rec, n)  # noqa: E731
    for i, root in enumerate(roots):
        T, sims = 2000 * n + i, sims_for[n]
        mc = (16, 4, 1, 1000, 8, 2)[i]
        R = 1 if i % 2 == 0 else 3
        noise = noise_for(n, 1, 100 * n + i)[0] if i % 3 else None
        # zero logits + host rollouts
        ref = spec.Search(root, SEED, T, R, sims, mc, gumbel=noise).run(sims)
        assert_harness_matches(harness_search(gh, root, n, T, R, sims, mc, noise), ref, n, (n, i, "rollouts"))
        # stand-in logits and values, other constants
        ref = spec.Search(root, SEED, T, 1, sims, mc, 20.0, 0.5, gumbel=noise).run(sims, stand_in_value, logit_fn)
        got = harness_search(gh, root, n, T, 1, sims, mc, noise, stand_in_value, logit_fn, 20.0, 0.5)
        assert_harness_matches(got, ref, n, (n, i, "stand-in"))


def test_bytes_per_tree(gh):
    # n = 12: 401 node slots of 448 + 16 + 22 * 120 bytes, 16 + 8 * 142 path bytes, 4 rollout slots of 448 + 16
    # bytes, 4 * 144 bytes of root noise
    assert gh.gh_bytes_per_tree(12, 400, 4) == 401 * (448 + 16 + 22 * 120) + 16 + 8 * 142 + 4 * (448 + 16) + 4 * 144


def test_gumbel_noise_on_cpu():
    import torch
    from twixt_for_open_spiel_b200.mcts import gumbel_noise
    g1 = torch.Generator().manual_seed(5)
    g2 = torch.Generator().manual_seed(5)
    a, b = gumbel_noise(64, 144, g1), gumbel_noise(64, 144, g2)
    assert a.dtype == torch.float32 and a.shape == (64, 144) and torch.equal(a, b)
    assert bool(torch.isfinite(a).all()) and abs(float(a.double().mean()) - 0.5772) < 0.05


# ---------------------------------------------------------------------------------------------- GPU ---
def _batch_with_roots(roots, n, extra=0):
    from twixt_for_open_spiel_b200 import TwixTBatch
    b = TwixTBatch(n, len(roots) + extra, 0, SEED)
    b.import_state(np.stack([r.export_record() for r in roots]), 0)
    return b


def _assert_matches(m, refs, n, tag):
    visits, sums, best = m.root_stats()
    action, policy = m.gumbel_stats()
    for t, ref in enumerate(refs):
        v, w, _ = ref.root_stats(n)
        ra, rp = ref.gumbel_stats(n)
        assert np.array_equal(visits[t], v), (tag, t)
        assert sums[t].tobytes() == w.tobytes(), (tag, t)
        assert action[t] == ra and best[t] == ra, (tag, t)
        assert policy[t].tobytes() == rp.tobytes(), (tag, t)


@pytest.mark.gpu
@pytest.mark.parametrize("n,trees,sims,R,mc,noisy", [(5, 36, 120, 1, 16, False), (5, 36, 120, 4, 4, True),
                                                     (8, 36, 80, 2, 16, True), (12, 24, 48, 1, 8, True),
                                                     (12, 24, 48, 4, 1, False), (24, 8, 24, 1, 16, True)])
def test_device_run_matches_spec(oracle_mod, n, trees, sims, R, mc, noisy):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 13 * n + R, trees)
    b = _batch_with_roots(roots, n)
    b.set_stream_base(500)
    m = BatchedMCTS(b, trees, sims, R, selection="gumbel", max_considered=mc)
    m.begin(0, trees)
    noise = noise_for(n, trees, n + R) if noisy else None
    if noisy:
        m.set_root_gumbel(noise)
    m.run(sims)
    refs = [spec.Search(r, SEED, 500 + t, R, sims, mc, gumbel=None if noise is None else noise[t]).run(sims)
            for t, r in enumerate(roots)]
    _assert_matches(m, refs, n, (n, R, mc))


def _stepwise(m, b, refs, n, trees, sims, device=False):
    import torch
    for k in range(sims):
        status = m.select(trees)
        leaves = b.export_state(trees, trees)
        values = np.zeros((trees, 2), dtype=np.float32)
        logits = np.zeros((trees, n * n), dtype=np.float32)
        for t, ref in enumerate(refs):
            leaf, terminal = ref.select()
            assert np.array_equal(leaves[t], ref.nodes[leaf].state.export_record()), (n, k, t)
            assert status[t] == int(terminal), (n, k, t)
            values[t] = stand_in_value(leaves[t])
            logits[t] = spec.stand_in_logits(leaves[t], n)
            ref.backup(values[t], logits[t])
        if device:
            m.backup(torch.from_numpy(values).cuda(), torch.from_numpy(logits).cuda())
        else:
            m.backup(values, logits)


@pytest.mark.gpu
@pytest.mark.parametrize("n,trees,sims,mc", [(5, 24, 60, 16), (8, 16, 40, 4), (12, 16, 32, 8), (24, 6, 20, 16)])
def test_stepwise_form_matches_spec(oracle_mod, n, trees, sims, mc):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 7 * n, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    noise = noise_for(n, trees, 3 * n)
    for device in (False, True):
        m = BatchedMCTS(b, trees, sims, 1, selection="gumbel", max_considered=mc, c_visit=30.0, c_scale=0.25)
        m.begin(0, trees)
        if device:
            import torch
            m.set_root_gumbel(torch.from_numpy(noise).cuda())
        else:
            m.set_root_gumbel(noise)
        refs = [spec.Search(r, SEED, t, 1, sims, mc, 30.0, 0.25, gumbel=noise[t]) for t, r in enumerate(roots)]
        _stepwise(m, b, refs, n, trees, sims, device)
        if device:
            import torch
            b.synchronize()
            act = torch.zeros(trees, dtype=torch.int32, device="cuda")
            pol = torch.zeros((trees, n * n), dtype=torch.float32, device="cuda")
            m.gumbel_stats(act, pol)
            b.synchronize()
            for t, ref in enumerate(refs):
                ra, rp = ref.gumbel_stats(n)
                assert int(act[t]) == ra and pol[t].cpu().numpy().tobytes() == rp.tobytes(), (n, t)
        _assert_matches(m, refs, n, (n, device))
        m.close()


@pytest.mark.gpu
def test_split_runs_sharded_roots_and_determinism(oracle_mod):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 64, 120
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 91, trees)
    b = _batch_with_roots(roots, n)
    before = b.export_state()
    noise = noise_for(n, trees, 4)
    m1 = BatchedMCTS(b, trees, sims, 2, selection="gumbel")
    m1.begin(0, trees)
    m1.set_root_gumbel(noise)
    m1.run(50)
    m1.run(70)
    split = m1.root_stats() + m1.gumbel_stats()
    m2 = BatchedMCTS(b, trees, sims, 2, selection="gumbel")
    for _ in range(2):
        m2.begin(0, trees)
        m2.set_root_gumbel(noise)
        m2.run(sims)
        whole = m2.root_stats() + m2.gumbel_stats()
        for x, y in zip(split, whole):
            assert x.tobytes() == y.tobytes()
    halves = []
    m3 = BatchedMCTS(b, trees // 2, sims, 2, selection="gumbel")
    for first in (0, trees // 2):
        m3.begin(first, trees // 2)
        m3.set_root_gumbel(noise[first:first + trees // 2])
        m3.run(sims)
        halves.append(m3.root_stats() + m3.gumbel_stats())
    for i in range(5):
        assert np.concatenate([halves[0][i], halves[1][i]]).tobytes() == whole[i].tobytes()
    assert b.export_state().tobytes() == before.tobytes()


@pytest.mark.gpu
def test_errors_budget_and_launch_counts(oracle_mod):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims = 8, 16, 30
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 19, trees)
    b = _batch_with_roots(roots, n, extra=trees)
    for kw in ({"max_considered": 0}, {"c_visit": float("nan")}, {"c_visit": -1.0}, {"c_scale": float("inf")},
               {"c_scale": -0.5}, {"solve": True}, {"leaves_per_step": 2}):
        with pytest.raises(ValueError):
            BatchedMCTS(b, trees, sims, 1, selection="gumbel", **kw)
    with pytest.raises(MemoryError, match="Gumbel MCTS arena"):
        BatchedMCTS(b, 1 << 40, 1000, 1, selection="gumbel")
    m = BatchedMCTS(b, trees, sims, 2, selection="gumbel")
    with pytest.raises(ValueError):
        m.gumbel_stats()  # before begin
    with pytest.raises(ValueError):
        m.set_root_gumbel(np.zeros((trees, n * n), dtype=np.float32))  # before begin
    m.begin(0, trees)
    noise = noise_for(n, trees, 8)
    bad = noise.copy()
    bad[2, 7] = np.inf
    with pytest.raises(ValueError, match="finite"):
        m.set_root_gumbel(bad)
    m.set_root_gumbel(noise)
    l0 = b.stats()["kernel_launches"]
    m.run(10)
    assert b.stats()["kernel_launches"] - l0 == 3 * 10
    refs = [spec.Search(r, SEED, t, 2, sims, 16, gumbel=noise[t]).run(10) for t, r in enumerate(roots)]
    _assert_matches(m, refs, n, "run")
    with pytest.raises(ValueError, match="Gumbel"):
        m.advance(np.full(trees, -1, dtype=np.int32))
    with pytest.raises(ValueError, match="Gumbel"):
        m.set_root_priors(np.full((trees, n * n), 1.0 / (n * n), dtype=np.float32))
    puct = BatchedMCTS(b, trees, sims, 2, selection="puct")
    puct.begin(0, trees)
    for call in (lambda: puct.set_root_gumbel(noise), lambda: puct.gumbel_stats()):
        with pytest.raises(ValueError, match="not a Gumbel search"):
            call()
    puct.close()
    for k in range(8):
        l0 = b.stats()["kernel_launches"]
        status = m.select(trees)
        launches = b.stats()["kernel_launches"] - l0
        leaves = b.export_state(trees, trees)
        values = np.stack([stand_in_value(r) for r in leaves])
        # finite on every legal cell and on a few illegal ones, -inf on the others
        logits = np.stack([spec.stand_in_logits(r, n) for r in leaves])
        legal = b.legal_mask(trees, trees).astype(bool)  # one launch of its own, not counted
        l0 = b.stats()["kernel_launches"]
        t_open = int(np.nonzero(status == 0)[0][0])
        legal_cell = int(np.nonzero(legal[t_open])[0][0])
        illegal_cell = int(np.nonzero(~legal[t_open])[0][0])
        for x in (np.nan, np.inf, -np.inf):
            junk = logits.copy()
            junk[t_open, legal_cell] = x
            with pytest.raises(ValueError, match="finite on the leaf's legal actions"):
                m.backup(values, junk)
        for call in (lambda: m.select(trees), lambda: m.run(1), lambda: m.gumbel_stats(),
                     lambda: m.set_root_gumbel(noise)):
            with pytest.raises(ValueError):
                call()
        logits[t_open, illegal_cell] = np.nan  # entries of illegal actions are ignored
        m.backup(values, logits)
        assert launches + b.stats()["kernel_launches"] - l0 == 2
        for t, ref in enumerate(refs):
            ref.select()
            ref.backup(values[t], logits[t])
    _assert_matches(m, refs, n, "after errors")
    l0 = b.stats()["kernel_launches"]
    m.gumbel_stats()
    assert b.stats()["kernel_launches"] - l0 == 1
    with pytest.raises(ValueError, match="max_simulations"):
        m.run(sims - 18 + 1)  # 18 simulations so far
    m.run(sims - 18)
    m.close()


@pytest.mark.gpu
def test_self_play_example():
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    try:
        import alphazero_selfplay
    finally:
        sys.path.pop(0)
    from twixt_for_open_spiel_b200 import load_game
    n, games, sims = 8, 32, 16
    trajectories, returns = alphazero_selfplay.self_play(n=n, games=games, sims=sims, seed=4, verbose=False,
                                                         search="gumbel", max_considered=8)
    game = load_game("twixt(board_size=%d)" % n)
    assert len(trajectories) == games and returns.shape == (games, 2)
    for gi, traj in enumerate(trajectories):
        state = game.new_initial_state()
        for step in traj:
            legal = np.zeros(n * n, dtype=bool)
            legal[state.legal_actions()] = True
            assert np.array_equal(step["mask"].astype(bool), legal), gi
            pol = step["policy"]
            assert abs(float(pol.sum(dtype=np.float64)) - 1.0) < 1e-5 and np.all(pol[~legal] == 0), gi
            assert legal[step["action"]], gi
            state.apply_action(int(step["action"]))
        assert state.is_terminal(), gi
        assert list(returns[gi]) == list(state.returns()), gi
    with pytest.raises(ValueError):
        alphazero_selfplay.self_play(n=n, games=4, sims=4, verbose=False, search="gumbel", reuse_tree=True)


@pytest.mark.gpu
def test_gumbel_search_at_scale():
    import torch
    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, gumbel_noise
    from twixt_for_open_spiel_b200.producer import ObservationMaskProducer
    n, trees, sims = 12, 8192, 32
    dev = torch.device("cuda:0")
    b = TwixTBatch(n, 2 * trees, 0, SEED)
    b.use_torch_stream()
    group = trees // 8
    for gi in range(8):
        b.playout(gi * group, group, max_plies=3 * gi, want_returns=False, want_lengths=False)
    producer = ObservationMaskProducer(b, max_count=trees)
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(12 * n * (n - 2), n * n + 1)).to(dev)
    m = BatchedMCTS(b, trees, sims, selection="gumbel", max_considered=16)
    m.begin(0, trees)
    m.set_root_gumbel(gumbel_noise(trees, n * n, device=dev))
    player = torch.zeros(trees, dtype=torch.int8, device=dev)
    with torch.no_grad():
        for _ in range(sims):
            m.select(trees)
            obs, mask = producer.produce(trees, trees)
            out = net(obs)
            logits = out[:, :n * n].masked_fill(~mask.bool(), float("-inf")).float().contiguous()
            v = torch.tanh(out[:, n * n])
            b.current_player(trees, trees, out=player)
            v = torch.where(player == 1, -v, v)
            m.backup(torch.stack([v, -v], dim=1).float().contiguous(), logits)
    visits, _, best = m.root_stats()
    action, policy = m.gumbel_stats()
    term = b.is_terminal(0, trees)
    mask = b.legal_mask(0, trees).astype(bool)
    assert np.array_equal(best, action)
    for t in range(trees):
        if term[t]:
            assert visits[t].sum() == 0 and action[t] == -1 and not policy[t].any()
        else:
            assert visits[t].sum() == sims - 1 and mask[t, action[t]] and visits[t, action[t]] == visits[t].max(), t
            assert abs(float(policy[t].sum(dtype=np.float64)) - 1.0) < 1e-5 and not policy[t][~mask[t]].any(), t
            assert np.count_nonzero(visits[t]) <= 16, t
