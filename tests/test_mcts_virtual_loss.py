"""Several leaves per step with virtual loss (twixt_mcts_create_parallel, BatchedMCTS(leaves_per_step=K)) against
its executable specification tests/vl_spec.py.  CPU: the specification's own properties, and the product's helpers
compiled for the host (tests/vl_harness.cc) node for node against it.  GPU: the device search bit for bit against
the specification (built-in rollouts and the stepwise form), K = 1 against twixt_mcts_create_ex, reproducibility,
host / device pointers, launch counts, errors, the bot and a search at scale."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import mcts_spec
import puct_spec
import vl_spec

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "twixt_for_open_spiel_b200", "csrc")
SEED = 0x766C6F73
KINDS = ["uct", "puct"]


def P(a):
    return a.ctypes.data_as(C.c_void_p)


def make(kind, root, seed, T, R=1, c=2.0, vl=1.0):
    cls = vl_spec.UctSearch if kind == "uct" else vl_spec.PuctSearch
    return cls(root, seed, T, R, c, vl)


def prior_fn(n):
    return lambda rec: puct_spec.stand_in_priors(rec, n)


def uct_dump(s):
    """Per node: (parent, action, N, L, [N(a)], [W(a)]) of a UCT specification."""
    return [(nd.parent, nd.action, nd.n, -1 if nd.actions is None else len(nd.actions), list(nd.edge_n),
             list(nd.edge_w)) for nd in s.nodes]


def dump(kind, s):
    return uct_dump(s) if kind == "uct" else s.dump()


# ------------------------------------------------------------------------------- the specification itself ---
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [5, 8, 12])
def test_spec_k1_is_the_base_search(oracle_mod, kind, n):
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 20 + n, 6)
    sims = {5: 60, 8: 40, 12: 24}[n]
    for i, root in enumerate(roots):
        R, T = 1 + i % 2, 100 * n + i
        if kind == "uct":
            ref = mcts_spec.Search(root, SEED, T, R, 1.5).run(sims)
            got = make(kind, root, SEED, T, R, 1.5).run_steps(sims, 1)
        else:
            ref = puct_spec.Search(root, SEED, T, R, 1.5).run(sims, None, prior_fn(n))
            got = make(kind, root, SEED, T, R, 1.5).run_steps(sims, 1, None, prior_fn(n))
        assert repr(dump(kind, got)) == repr(dump(kind, ref)), (kind, n, i)
        assert got.root_stats(n)[2] == ref.root_stats(n)[2]


@pytest.mark.parametrize("kind", KINDS)
def test_spec_virtual_counts_vanish_and_step0_stops_at_the_root(oracle_mod, kind):
    n, K = 8, 7
    g = oracle_mod.OracleGame(n)
    for i, root in enumerate(mcts_spec.root_positions(g, n, 4, 6)):
        s = make(kind, root, SEED, i, 1, 2.0, 0.5)
        for step in range(12):
            leaves = s.select_step(K)
            if step == 0:
                assert [leaf for leaf, _ in leaves] == [0] * K
            vals = [None if t else mcts_spec.stand_in_value(s.nodes[leaf].state.export_record()) for leaf, t in leaves]
            pri = [None if t else puct_spec.stand_in_priors(s.nodes[leaf].state.export_record(), n)
                   for leaf, t in leaves]
            s.backup_step(vals, pri)
            assert not any(s.virtual_counts()), (kind, i, step)
        assert s.k == 12 * K


def test_spec_uct_step1_reaches_k_distinct_new_children(oracle_mod):
    n = 8
    g = oracle_mod.OracleGame(n)
    root = g.new_initial_state()
    for K in (2, 7, 32):
        s = make("uct", root, SEED, K)
        s.run_steps(K, K, mcts_spec.stand_in_value)
        leaves = s.select_step(K)
        assert len(root.legal_actions()) >= K
        assert len({leaf for leaf, _ in leaves}) == K
        assert all(s.nodes[leaf].parent == 0 and s.nodes[leaf].n == 0 for leaf, _ in leaves)
        assert len(s.nodes) == 1 + K


def test_spec_hand_traced_two_steps(oracle_mod):
    """n = 5, UCT, K = 3, vl = 1, value +0.5 for player 0 on every leaf.  Step 0: three rows at the root, so
    N(root) = 3 and the root has no edges yet.  Step 1: the root is expanded (L edges, all unvisited); descent 0
    draws among L edges with k = 3, descent 1 among the L - 1 with V = 0 with k = 4, descent 2 among L - 2 with
    k = 5; each creates one child.  After the backup every taken edge has N = 1 and W = v[0] = 0.5."""
    n, K = 5, 3
    g = oracle_mod.OracleGame(n)
    root = g.new_initial_state()
    s = make("uct", root, SEED, 9)
    half = np.asarray([0.5, -0.5], dtype=np.float32)
    assert s.select_step(K) == [(0, False)] * K
    s.backup_step([half] * K)
    assert s.nodes[0].n == 3 and s.nodes[0].actions is None and s.k == 3
    leaves = s.select_step(K)
    legal = root.legal_actions()
    free = list(range(len(legal)))
    expect = []
    for j in range(K):
        e = free.pop(mcts_spec.draw(SEED, 9, 3 + j, len(free)))
        expect.append(e)
    assert [s.nodes[leaf].action for leaf, _ in leaves] == [legal[e] for e in expect]
    assert s.ve[0] == [1 if i in expect else 0 for i in range(len(legal))] and s.vn[0] == K
    s.backup_step([half] * K)
    assert s.nodes[0].n == 6 and s.k == 6
    for i in range(len(legal)):
        assert (s.nodes[0].edge_n[i], s.nodes[0].edge_w[i]) == ((1, 0.5) if i in expect else (0, 0.0))
    # step 2: every visited edge has n_eff >= 1, so descent 0 still draws among the L - 3 unvisited edges
    leaves = s.select_step(K)
    assert all(s.nodes[leaf].parent == 0 and s.nodes[leaf].n == 0 for leaf, _ in leaves)
    assert len({leaf for leaf, _ in leaves}) == K


def test_spec_virtual_loss_spreads_puct_descents(oracle_mod):
    """With a large virtual loss the K descents of a step avoid each other's edges at the root."""
    n, K = 8, 8
    g = oracle_mod.OracleGame(n)
    root = g.new_initial_state()
    s = make("puct", root, SEED, 3, 1, 2.0, 100.0)
    s.run_steps(K, K, mcts_spec.stand_in_value, prior_fn(n))
    leaves = s.select_step(K)
    assert len({leaf for leaf, _ in leaves}) == K


# ----------------------------------------------------------------------- host harness vs specification ---
@pytest.fixture(scope="module")
def vh():
    out_dir = os.path.join(HERE, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libvlharness.so")
    src = os.path.join(HERE, "vl_harness.cc")
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-x", "c++", "-fPIC",
                               "-shared", "-I", CSRC, "-o", so, src])
    lib = C.CDLL(so)
    lib.vh_bytes_per_tree.restype = C.c_int64
    lib.vh_bytes_per_tree.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.vh_create.restype = C.c_void_p
    lib.vh_create.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_double, C.c_int, C.c_int,
                              C.c_int, C.c_double]
    lib.vh_destroy.argtypes = [C.c_void_p]
    lib.vh_select_step.restype = C.c_int
    lib.vh_select_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.vh_backup_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.vh_dump.restype = C.c_int
    lib.vh_dump.argtypes = [C.c_void_p] + [C.c_void_p] * 10
    return lib


def harness_check(vh, kind, root, n, T, R, c, vl, sims, K, stand_in):
    """Runs the harness and the specification in lock step (values from host rollouts or stand-ins) and compares
    every node after every step: N(s), V(s), edge count, N(a), W(a) bit for bit, V(a) and (PUCT) P(a)."""
    rec = np.ascontiguousarray(root.export_record())
    rw = rec.size
    h = vh.vh_create(P(rec), n, SEED, T, R, c, sims, 1 if kind == "puct" else 0, K, vl)
    ref = make(kind, root, SEED, T, R, c, vl)
    S, M = sims + 1, n * (n - 2)
    leaves_out = np.zeros((K, rw), dtype=np.uint32)
    leaf_slot = np.zeros(K, dtype=np.int32)
    status = np.zeros(K, dtype=np.int32)
    arrays = dict(parent=np.zeros(S, np.int32), action=np.zeros(S, np.int32), nn=np.zeros(S, np.uint32),
                  nv=np.zeros(S, np.uint32), legal=np.zeros(S, np.int32), en=np.zeros((S, M), np.uint32),
                  ew=np.zeros((S, M), np.float64), ev=np.zeros((S, M), np.uint32), ep=np.zeros((S, M), np.float32),
                  best=np.zeros(1, np.int32))
    try:
        for step in range(sims // K):
            count = vh.vh_select_step(h, P(leaves_out), P(leaf_slot), P(status))
            got = ref.select_step(K)
            assert [(int(a), bool(b)) for a, b in zip(leaf_slot, status)] == got, (kind, n, T, step)
            assert count == len(ref.nodes)
            vals = np.zeros((K, 2), dtype=np.float32)
            pri = np.zeros((K, n * n), dtype=np.float32)
            spec_vals, spec_pri = [], []
            for j, (leaf, terminal) in enumerate(got):
                r = leaves_out[j]
                assert np.array_equal(r, ref.nodes[leaf].state.export_record())
                if terminal:
                    spec_vals.append(None)
                elif stand_in:
                    vals[j] = mcts_spec.stand_in_value(r)
                    spec_vals.append(vals[j])
                else:
                    v = ref.rollout_value_at(leaf, ref.k + j)
                    spec_vals.append(v)
                pri[j] = puct_spec.stand_in_priors(r, n)
                spec_pri.append(None if terminal or not stand_in else pri[j])
            vh.vh_backup_step(h, P(vals) if stand_in else None, P(pri) if stand_in else None)
            ref.backup_step(spec_vals, spec_pri)
            a = arrays
            nodes = vh.vh_dump(h, P(a["parent"]), P(a["action"]), P(a["nn"]), P(a["nv"]), P(a["legal"]), P(a["en"]),
                               P(a["ew"]), P(a["ev"]), P(a["ep"]), P(a["best"]))
            d = dump(kind, ref)
            assert nodes == len(d)
            assert not a["nv"][:nodes].any() and not a["ev"][:nodes].any()
            for s_, row in enumerate(d):
                par, act, nn, L, e_n, e_w = row[:6]
                assert (a["parent"][s_], a["action"][s_], a["nn"][s_], a["legal"][s_]) == (par, act, nn, L), \
                    (kind, n, T, step, s_)
                if L > 0:
                    assert a["en"][s_, :L].tolist() == e_n
                    assert a["ew"][s_, :L].tobytes() == np.asarray(e_w, dtype=np.float64).tobytes()
                    if kind == "puct":
                        assert a["ep"][s_, :L].tobytes() == np.asarray(row[6], dtype=np.float32).tobytes()
        assert int(a["best"][0]) == ref.root_stats(n)[2]
    finally:
        vh.vh_destroy(h)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [5, 8, 12])
@pytest.mark.parametrize("K", [1, 2, 7, 32])
def test_harness_matches_spec_node_for_node(vh, oracle_mod, kind, n, K):
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 70 + n + K, 6)
    sims = {5: 64, 8: 64, 12: 32}[n]
    sims = max(K, sims - sims % K) if K > 1 else sims
    if K == 32:
        sims = 96 if n < 12 else 64
    for i, root in enumerate(roots):
        vl = (1.0, 0.5, 3.0)[i % 3]
        harness_check(vh, kind, root, n, 2000 * n + i, 1 + (i % 2) * 2, (2.0, 0.7)[i % 2], vl, sims, K,
                      stand_in=i % 2 == 1)


def test_bytes_per_tree_formula(vh):
    # n = 12, 400 simulations, R = 4: the UCT arena plus (K - 1) * (16 + 8*142 + 4*(448 + 16)) + 401 * 2 * (1 + 120)
    base = 401 * (448 + 8 + 18 * 120) + 16 + 8 * 142 + 4 * (448 + 16)
    assert vh.vh_bytes_per_tree(12, 400, 4, 0, 1) == base
    assert vh.vh_bytes_per_tree(12, 400, 4, 0, 8) == base + 7 * (16 + 8 * 142 + 4 * 464) + 401 * 2 * 121
    assert vh.vh_bytes_per_tree(12, 400, 4, 1, 8) == base + 401 * 9 * 120 + 7 * (16 + 8 * 142 + 4 * 464) + \
        401 * 2 * 121


# ---------------------------------------------------------------------------------------------- GPU ---
def _batch_with_roots(roots, n, extra=0, seed=SEED):
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


class _Counted:
    """Counts the plies and games of a specification's rollouts (what twixt_stats must add)."""

    def __init__(self):
        self.plies = 0
        self.games = 0

    def wrap(self, s):
        orig = s.rollout_value_at

        def rollout_value_at(leaf, k):
            for r in range(s.R):
                st = s.nodes[leaf].state.clone()
                self.plies += len(st.playout_philox(s.seed, mcts_spec.rollout_stream(s.T, k, s.R, r)))
                self.games += 1
            return orig(leaf, k)
        s.rollout_value_at = rollout_value_at
        return s


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,trees,sims", [(5, 24, 96), (8, 24, 64), (12, 16, 48), (24, 8, 32)])
@pytest.mark.parametrize("K", [1, 4, 16])
def test_device_run_matches_spec(oracle_mod, kind, n, trees, sims, K):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 17 * n + K, trees)
    R = 2
    b = _batch_with_roots(roots, n)
    b.set_stream_base(700)
    m = BatchedMCTS(b, trees, sims, R, 1.25, selection=kind, leaves_per_step=K, virtual_loss=0.75)
    m.begin(0, trees)
    b.stats_reset()
    l0 = b.stats()["kernel_launches"]
    m.run(sims)
    assert b.stats()["kernel_launches"] - l0 == 3 * (sims // K)
    counter = _Counted()
    refs = [counter.wrap(make(kind, r, SEED, 700 + t, R, 1.25, 0.75)).run_steps(sims, K)
            for t, r in enumerate(roots)]
    _assert_stats_equal(m.root_stats(), refs, n, (kind, n, K))
    st = b.stats()
    assert (st["plies"], st["games"]) == (counter.plies, counter.games), (kind, n, K)


def _stepwise(m, b, refs, n, trees, K, steps, device=False, check_leaves=True):
    """Drives the device search and the specification in lock step with stand-in values and priors."""
    import torch
    n_rows = trees * K
    for step in range(steps):
        status = m.select(trees)
        leaves = b.export_state(trees, n_rows)
        values = np.zeros((n_rows, 2), dtype=np.float32)
        priors = np.zeros((n_rows, n * n), dtype=np.float32)
        for t, ref in enumerate(refs):
            got = ref.select_step(K)
            vals, pri = [], []
            for j, (leaf, terminal) in enumerate(got):
                row = t * K + j
                if check_leaves:
                    assert np.array_equal(leaves[row], ref.nodes[leaf].state.export_record()), (n, step, t, j)
                    assert status[row] == int(terminal), (n, step, t, j)
                values[row] = mcts_spec.stand_in_value(leaves[row])
                priors[row] = puct_spec.stand_in_priors(leaves[row], n)
                vals.append(None if terminal else values[row])
                pri.append(None if terminal else priors[row])
            ref.backup_step(vals, pri)
        if device:
            m.backup(torch.from_numpy(values).cuda(), torch.from_numpy(priors).cuda())
        else:
            m.backup(values, priors if m.selection == "puct" else None)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,trees,sims", [(5, 12, 64), (8, 12, 48), (12, 8, 32), (24, 4, 32)])
@pytest.mark.parametrize("K", [1, 4, 16])
def test_stepwise_form_matches_spec(oracle_mod, kind, n, trees, sims, K):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 3 * n + K, trees)
    b = _batch_with_roots(roots, n, extra=trees * K)
    m = BatchedMCTS(b, trees, sims, 1, 2.0, selection=kind, leaves_per_step=K, virtual_loss=1.5)
    m.begin(0, trees)
    refs = [make(kind, r, SEED, t, 1, 2.0, 1.5) for t, r in enumerate(roots)]
    l0 = b.stats()["kernel_launches"]
    _stepwise(m, b, refs, n, trees, K, sims // K)
    assert b.stats()["kernel_launches"] - l0 == 2 * (sims // K)
    _assert_stats_equal(m.root_stats(), refs, n, (kind, n, K))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_k1_parallel_is_create_ex(oracle_mod, kind):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, _PUCT
    n, trees, sims = 8, 32, 60
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 31, trees)
    b = _batch_with_roots(roots, n)
    out = []
    for parallel in (False, True):
        m = BatchedMCTS(b, trees, sims, 2, selection=kind)
        if parallel:  # the same search made with twixt_mcts_create_parallel(K = 1)
            m.close()
            m._check(m._lib.twixt_mcts_create_parallel(b._h, trees, sims, 2, 2.0, _PUCT if kind == "puct" else 0,
                                                       1, 5.0, C.byref(m._h)))
        m.begin(0, trees)
        l0 = b.stats()["kernel_launches"]
        m.run(sims)
        assert b.stats()["kernel_launches"] - l0 == 3 * sims
        out.append(m.root_stats())
        m.close()
    for x, y in zip(*out):
        assert x.tobytes() == y.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_reproducibility_split_runs_and_sharded_roots(oracle_mod, kind):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, K = 8, 8
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 78, 64)
    b = _batch_with_roots(roots, n)
    before = b.export_state()
    m1 = BatchedMCTS(b, 64, 200, 2, selection=kind, leaves_per_step=K)
    m1.begin(0, 64)
    m1.run(64)
    m1.run(136)
    split = m1.root_stats()
    m2 = BatchedMCTS(b, 64, 200, 2, selection=kind, leaves_per_step=K)
    m2.begin(0, 64)
    m2.run(200)
    whole = m2.root_stats()
    for x, y in zip(split, whole):
        assert x.tobytes() == y.tobytes()
    halves = []
    m3 = BatchedMCTS(b, 32, 200, 2, selection=kind, leaves_per_step=K)
    for first in (0, 32):
        m3.begin(first, 32)
        m3.run(200)
        halves.append(m3.root_stats())
    for i in range(3):
        assert np.concatenate([halves[0][i], halves[1][i]]).tobytes() == whole[i].tobytes()
    assert b.export_state().tobytes() == before.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_host_and_device_pointers_give_identical_trees(oracle_mod, kind):
    import torch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, K, sims = 8, 16, 4, 40
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 8, trees)
    b = _batch_with_roots(roots, n, extra=trees * K)
    out = []
    for device in (False, True):
        m = BatchedMCTS(b, trees, sims, 1, selection=kind, leaves_per_step=K)
        m.begin(0, trees)
        refs = [make(kind, r, SEED, t) for t, r in enumerate(roots)]
        _stepwise(m, b, refs, n, trees, K, sims // K, device=device and kind == "puct")
        out.append(m.root_stats())
        _assert_stats_equal(out[-1], refs, n, device)
        m.close()
    for x, y in zip(*out):
        assert x.tobytes() == y.tobytes()
    # torch tensors on torch's stream, statuses and outputs on the device
    b.use_torch_stream()
    m = BatchedMCTS(b, trees, sims, 1, selection=kind, leaves_per_step=K)
    m.begin(0, trees)
    status = torch.zeros(trees * K, dtype=torch.int32, device="cuda")
    refs = [make(kind, r, SEED, t) for t, r in enumerate(roots)]
    for _ in range(sims // K):
        m.select(trees, status)
        leaves = b.export_state(trees, trees * K)
        vals = np.stack([mcts_spec.stand_in_value(r) for r in leaves])
        pri = np.stack([puct_spec.stand_in_priors(r, n) for r in leaves])
        for t, ref in enumerate(refs):
            got = ref.select_step(K)
            ref.backup_step([None if term else vals[t * K + j] for j, (_, term) in enumerate(got)],
                            [None if term else pri[t * K + j] for j, (_, term) in enumerate(got)])
        m.backup(torch.from_numpy(vals).cuda(), torch.from_numpy(pri).cuda() if kind == "puct" else None)
    torch.cuda.current_stream().synchronize()
    assert status.cpu().numpy().min() >= 0
    dev = (torch.zeros((trees, n * n), dtype=torch.int32, device="cuda"),
           torch.zeros((trees, n * n), dtype=torch.float64, device="cuda"),
           torch.zeros(trees, dtype=torch.int32, device="cuda"))
    m.root_stats(*dev)
    torch.cuda.current_stream().synchronize()
    _assert_stats_equal([x.cpu().numpy() for x in dev], refs, n, "torch")


@pytest.mark.gpu
def test_errors_leave_the_search_exact(oracle_mod):
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, K, sims = 8, 8, 4, 40
    g = oracle_mod.OracleGame(n)
    roots = mcts_spec.root_positions(g, n, 19, trees)
    b = _batch_with_roots(roots, n, extra=trees * K)
    for bad in (dict(leaves_per_step=0), dict(leaves_per_step=4097), dict(leaves_per_step=-3),
                dict(leaves_per_step=41), dict(leaves_per_step=4, virtual_loss=float("nan")),
                dict(leaves_per_step=4, virtual_loss=-0.5), dict(leaves_per_step=4, virtual_loss=float("inf")),
                dict(leaves_per_step=2, solve=True), dict(leaves_per_step=2, selection="puct", solve=True)):
        with pytest.raises(ValueError):
            BatchedMCTS(b, trees, sims, 2, **bad)
    with pytest.raises(ValueError, match="leaves_per_step"):
        BatchedMCTS(b, trees, sims, 2, leaves_per_step=5000)
    with pytest.raises(ValueError, match="virtual_loss"):
        BatchedMCTS(b, trees, sims, 2, leaves_per_step=2, virtual_loss=float("nan"))
    with pytest.raises(MemoryError, match="leaves per step"):
        BatchedMCTS(b, 1 << 36, 1000, 1, leaves_per_step=8)
    m = BatchedMCTS(b, trees, sims, 2, selection="puct", leaves_per_step=K)
    m.begin(0, trees)
    refs = [make("puct", r, SEED, t, 2) for t, r in enumerate(roots)]
    for call in (lambda: m.run(K + 1), lambda: m.run(1), lambda: m.select(trees + 1),
                 lambda: m.select(b.num_envs - trees * K + 1)):
        with pytest.raises(ValueError):
            call()
    m.run(2 * K)
    for ref in refs:
        ref.run_steps(2 * K, K)
    _assert_stats_equal(m.root_stats(), refs, n, "run")
    cells = n * n
    for step in range(3):
        status = m.select(trees)
        assert status.shape == (trees * K,)
        leaves = b.export_state(trees, trees * K)
        values = np.stack([mcts_spec.stand_in_value(r) for r in leaves])
        priors = np.stack([puct_spec.stand_in_priors(r, n) for r in leaves])
        for x in (float("nan"), -1e-3, float("inf")):
            p = priors.copy()
            p[trees * K - 1, cells - 1] = x  # the last row: the check covers all count*K rows
            with pytest.raises(ValueError):
                m.backup(values, p)
        with pytest.raises(ValueError):
            m.run(K)
        m.backup(values, priors)
        for t, ref in enumerate(refs):
            got = ref.select_step(K)
            ref.backup_step([None if term else values[t * K + j] for j, (_, term) in enumerate(got)],
                            [None if term else priors[t * K + j] for j, (_, term) in enumerate(got)])
    _assert_stats_equal(m.root_stats(), refs, n, "after errors")
    with pytest.raises(ValueError):
        m.run(sims)  # beyond max_simulations


@pytest.mark.gpu
def test_bot_plays_a_legal_game_with_8_leaves_per_step():
    from twixt_for_open_spiel_b200 import load_game
    from twixt_for_open_spiel_b200.mcts import MCTSBot
    game = load_game("twixt(board_size=8)")
    bot = MCTSBot(game, max_simulations=200, n_rollouts=2, seed=5, leaves_per_step=8)
    state = game.new_initial_state()
    while not state.is_terminal():
        a = bot.step(state)
        assert a in state.legal_actions()
        state.apply_action(a)
    assert state.is_terminal()
    bot.close()
    with pytest.raises(ValueError):
        MCTSBot(game, max_simulations=100, leaves_per_step=8)


@pytest.mark.gpu
def test_virtual_loss_search_at_scale():
    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    n, trees, sims, K = 12, 8192, 400, 4
    b = TwixTBatch(n, trees, 0, SEED)
    b.use_torch_stream()
    group = trees // 8
    for gi in range(8):
        b.playout(gi * group, group, max_plies=3 * gi, want_returns=False, want_lengths=False)
    m = BatchedMCTS(b, trees, sims, 4, leaves_per_step=K)
    m.begin(0, trees)
    l0 = b.stats()["kernel_launches"]
    m.run(sims)
    assert b.stats()["kernel_launches"] - l0 == 3 * sims // K
    visits, _, best = m.root_stats()
    term = b.is_terminal(0, trees)
    for t in range(trees):
        if term[t]:
            assert visits[t].sum() == 0 and best[t] == -1
        else:
            assert visits[t].sum() == sims - K and best[t] >= 0 and visits[t, best[t]] > 0, t
