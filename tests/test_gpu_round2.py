"""-m gpu, second batch: every compiled playout kernel against the oracle, the CUDA path against the COMPILED
REFERENCE directly, BASELINE config C2 at its stated size, import validation, the bounds-instrumented
variant of the playout kernel, the fused observation+mask producer, device-side history replay and ToString
on records that came out of the CUDA path."""
import json
import os
import random
import subprocess
import sys
import textwrap
import zlib

import numpy as np
import pytest

from helpers import SEED, Digest, golden_digests, pad_games, random_game_actions

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


# ---------------------------------------------------------------- K5, every compiled size ---
@pytest.mark.parametrize("n", list(range(5, 25)))
def test_fused_playout_every_board_size(oracle_mod, n):
    """playout_kernel<N> is a separate binary kernel for every N = 5..24: 1 024 complete games at each size,
    every final record, return and length equal to the oracle's replay of the same Philox stream
    (twixtboard.cc:457-499 per move, 537-588 for the border flags, 192-207 for the result)."""
    from twixt_for_open_spiel_b200 import TwixTBatch
    og = oracle_mod.OracleGame(n)
    E = 1024
    batch = TwixTBatch(n, E, 0, SEED + n)
    batch.set_stream_base(10_000 * n)
    rets, lens, _ = batch.playout()
    recs = batch.export_state()
    st = batch.stats()
    assert st["games"] == E and st["plies"] == int(lens.sum()) and st["debug_violations"] == 0
    assert st["red_wins"] + st["blue_wins"] + st["draws"] == E
    want_recs = np.zeros_like(recs)
    want_rets = np.zeros_like(rets)
    want_lens = np.zeros_like(lens)
    outcomes = set()
    for e in range(E):
        s = og.new_initial_state()
        want_lens[e] = len(s.playout_philox(SEED + n, 10_000 * n + e))
        want_rets[e] = s.returns()
        want_recs[e] = s.export_record()
        outcomes.add(tuple(s.returns()))
    assert np.array_equal(lens, want_lens), n
    assert np.array_equal(rets, want_rets), n
    assert np.array_equal(recs, want_recs), n
    assert len(outcomes) >= 2  # wins (with their floods) and draws both occurred at this size
    batch.close()


# ------------------------------------------------------------ CUDA vs the compiled reference ---
def ref_worker_games(n):  # (lock-step games, fused playouts) per board size
    return (24, 256) if n <= 12 else (8, 128)


def _ref_worker(n, lock_games, fused):
    res = subprocess.run([sys.executable, os.path.join(HERE, "ref_gpu_worker.py"), str(n), str(lock_games), str(fused)],
                         capture_output=True, text=True, timeout=1500)
    assert res.returncode == 0 and "ref-direct ok" in res.stdout, (res.stdout[-500:], res.stderr[-3000:])


@pytest.mark.parametrize("n", list(range(5, 25)))
def test_cuda_against_compiled_reference(oracle_mod, n):
    """The parity chain closed on ONE machine: CUDA <-> oracle/_ref/libtwixt_ref.so (the unmodified reference,
    compiled in the authoring container, shipped to this box), lock-step and fused playouts, one process per
    board size because of the reference's static BlockerMap (twixtboard.cc:148-165,211).  Without oracle/_ref the
    worker compares with the stored digests of the reference's outputs on the same games."""
    _ref_worker(n, *ref_worker_games(n))


def playthrough_ply_digests(new_state, to_string):
    """Per ply of the golden playthrough (n = 8): a digest of every observable and the ToString picture."""
    with open(os.path.join(HERE, "golden", "playthrough_n8.json")) as f:
        actions = json.load(f)["actions"]
    st = new_state()
    out = []
    for ply in range(36):
        out.append(Digest().add(st.legal_actions(), st.current_player(), st.is_terminal(), st.returns(),
                                np.asarray(st.observation_tensor(0), dtype=np.float32),
                                np.asarray(st.export_record(), dtype=np.uint32), to_string(st)).hex())
        if ply < 35:
            st.apply_action(actions[ply])
    return out


def test_cuda_playthrough_against_compiled_reference_in_process(oracle_mod):
    """The golden playthrough (n = 8) with the CUDA adapter and the compiled reference side by side in THIS
    process: every ply, every observable, and the ToString picture of the CUDA-exported record.  Without
    oracle/_ref, every ply is compared with the stored digest of the reference's observables there."""
    from twixt_for_open_spiel_b200 import load_game
    with open(os.path.join(HERE, "golden", "playthrough_n8.json")) as f:
        pt = json.load(f)
    got = playthrough_ply_digests(load_game("twixt").new_initial_state, lambda st: st.to_string())
    want = golden_digests()["playthrough"]
    for ply in range(36):
        assert got[ply] == want[ply], ply
    if not oracle_mod.have_reference():
        return
    rg = oracle_mod.RefGame(8, True)
    rs = rg.new_initial_state()
    st = load_game("twixt").new_initial_state()
    by_index = {s["index"]: s for s in pt["states"]}
    strings = 0
    for ply in range(36):
        assert st.legal_actions() == rs.legal_actions() and st.current_player() == rs.current_player()
        assert st.is_terminal() == rs.is_terminal() and st.returns() == rs.returns()
        assert np.array_equal(np.asarray(st.observation_tensor(0), dtype=np.float32), rs.observation_tensor(0))
        assert np.array_equal(st.export_record(), rs.export_record())
        assert st.to_string() == rs.to_string()
        s = by_index.get(ply)
        if s is not None and "observation_string" in s:  # the 9 dumped states of playthrough.txt
            assert st.observation_string(0) == s["observation_string"]
            assert st.information_state_string(1) == s["observation_string"]
            strings += 1
        if ply < 35:
            st.apply_action(pt["actions"][ply])
            rs.apply_action(pt["actions"][ply])
    assert strings >= 9 and st.to_string().endswith("[x has won]")
    del rs, rg


def test_to_string_on_cuda_records_reference_fixture():
    """ToString at EVERY ply of the reference-generated string fixture (swap, both wins, draw, links of all
    eight directions in both colours, ANSI on/off), rendered from records exported by the CUDA path."""
    from twixt_for_open_spiel_b200 import load_game
    with open(os.path.join(HERE, "golden", "ref_strings.json")) as f:
        games = json.load(f)["games"]
    for g in games:
        game = load_game("twixt", {"board_size": g["n"], "ansi_color_output": g["ansi"]})
        st = game.new_initial_state()
        for ply in range(len(g["actions"]) + 1):
            text = st.to_string()
            assert zlib.crc32(text.encode("utf-8")) & 0xFFFFFFFF == g["crcs"][ply], (g["n"], g["ansi"], ply)
            if str(ply) in g["strings"]:
                assert text == g["strings"][str(ply)]
            if ply < len(g["actions"]):
                st.apply_action(g["actions"][ply])
        assert st.returns() == g["returns"]


# ----------------------------------------------------------------- BASELINE config C2 ---
def test_n5_differential_at_config_c2_size(oracle_mod):
    """BASELINE.json configs[1] at its stated size: all 15 first moves x {swap where legal, 2-3 other replies} x 10 000
    random continuations = 450 000 games at n = 5 in ONE batch.  Every continuation is regenerated by the
    oracle from the same prefix (trace, length, returns, final record); 45 x 40 of them are then replayed in
    lock-step with every observable compared at every ply."""
    from test_gpu_parity import _lockstep
    from twixt_for_open_spiel_b200 import TwixTBatch
    n, per = 5, 10_000
    og = oracle_mod.OracleGame(n)
    rng = random.Random(55)
    first_moves = og.new_initial_state().legal_actions()
    assert len(first_moves) == 15
    groups = []
    for f in first_moves:
        st = og.new_initial_state()
        st.apply_action(f)
        replies = st.legal_actions()
        # the swap offer where the cell is in blue's list (twixtboard.cc:485-488: not on rows 0 / n-1), + others
        others = rng.sample([a for a in replies if a != f], 3)
        for r in ([f] + others[:2]) if f in replies else others:
            groups.append((f, r))
    assert sum(1 for f, r in groups if f == r) == 9  # 3 columns x 3 inner rows
    E = len(groups) * per
    assert E == 450_000
    batch = TwixTBatch(n, E, 0, SEED)
    a0 = np.repeat(np.array([g[0] for g in groups], dtype=np.int32), per)
    a1 = np.repeat(np.array([g[1] for g in groups], dtype=np.int32), per)
    batch.apply(a0)
    batch.apply(a1)
    rets, lens, trace = batch.playout(trace=True)
    recs = batch.export_state()
    assert bool(batch.is_terminal().all())
    results = set()
    lock_games = []
    for gi, (f, r) in enumerate(groups):
        prefix = og.new_initial_state()
        prefix.apply_action(f)
        prefix.apply_action(r)
        want_recs = np.zeros((per, recs.shape[1]), dtype=np.uint32)
        want_rets = np.zeros((per, 2), dtype=np.float32)
        for j in range(per):
            e = gi * per + j
            s = prefix.clone()
            acts = s.playout_philox(SEED, e)
            assert lens[e] == len(acts) and trace[:lens[e], e].tolist() == acts, (f, r, j)
            want_recs[j] = s.export_record()
            want_rets[j] = s.returns()
            if j < 40:
                lock_games.append([f, r] + acts)
        assert np.array_equal(recs[gi * per:(gi + 1) * per], want_recs), (f, r)
        assert np.array_equal(rets[gi * per:(gi + 1) * per], want_rets), (f, r)
        results |= {tuple(x) for x in np.unique(want_rets, axis=0).tolist()}
    assert results == {(1.0, -1.0), (-1.0, 1.0), (0.0, 0.0)}  # red wins, blue wins and draws all occurred
    st = batch.stats()
    assert st["swaps"] == 0 and st["games"] == E  # the swaps here were made by twixt_apply, not by the playout
    batch.close()
    _lockstep(oracle_mod, n, lock_games)


# ------------------------------------------------------------------- import validation ---
def _mid_game_records(n, count, seed):
    from twixt_for_open_spiel_b200 import TwixTBatch
    b = TwixTBatch(n, count, 0, seed)
    for e in range(count):  # envs at different depths, some swapped, some finished
        b.playout(e, 1, max_plies=(e * 7) % (n * n), want_returns=False, want_lengths=False)
    recs = b.export_state()
    b.close()
    return recs


@pytest.mark.parametrize("n", [5, 6, 8, 13, 24])
def test_import_state_validates_records(oracle_mod, n):
    """twixt_import_state refuses records no sequence of legal moves can produce (the reference only reaches
    states through DoApplyAction, twixt.h:93-104) and leaves the batch untouched; reachable records pass."""
    from twixt_for_open_spiel_b200 import TwixTBatch
    E = 96
    good = _mid_game_records(n, E, SEED + 3)
    rw = good.shape[1]
    batch = TwixTBatch(n, E, 0, SEED)
    batch.import_state(good)  # every reachable record is accepted
    assert np.array_equal(batch.export_state(), good)
    init = oracle_mod.OracleGame(n).new_initial_state().export_record()
    batch.reset()
    P = lambda plane, col: 4 + plane * n + col  # noqa: E731
    has_link = [e for e in range(E) if good[e, P(2, 0):P(6, 0)].any()]
    busy = max(range(E), key=lambda e: int(good[e, 0]) * int((good[e, 1] & 3) == 0))  # deepest open game
    assert has_link and good[busy, 0] > 4

    def corrupt(e, fn):
        bad = good.copy()
        fn(bad[e])
        return bad, e

    def add_red_in_blue_end_column(r):
        r[P(0, n - 1)] |= 2

    def clear_one_peg(r):  # a peg vanishes: counts, links and flags no longer fit
        col = next(c for c in range(n) if r[P(0, c)] | r[P(1, c)])
        plane = 0 if r[P(0, col)] else 1
        r[P(plane, col)] &= r[P(plane, col)] - 1

    def link_without_peg(r):  # (no empty cell left in those columns: the record stays as it is and the case is skipped)
        for c in range(n - 2):
            free = ~int(r[P(0, c)] | r[P(1, c)]) & ((1 << (n - 1)) - 2)
            if free:
                r[P(2, c)] |= free & -free
                return

    cases = [
        ("header", corrupt(busy, lambda r: r.__setitem__(1, 8))),
        ("header", corrupt(busy, lambda r: r.__setitem__(0, n * n))),
        ("rows", corrupt(busy, lambda r: r.__setitem__(P(0, 1), r[P(0, 1)] | (1 << n)))),
        ("pegs", corrupt(busy, add_red_in_blue_end_column)),
        ("pegs", corrupt(busy, lambda r: r.__setitem__(P(1, 2), r[P(1, 2)] | r[P(0, 2)] | 1))),  # blue on row 0 / overlap
        ("counts", corrupt(busy, lambda r: r.__setitem__(3, r[3] + 1))),
        ("", corrupt(busy, clear_one_peg)),
        ("first-move", corrupt(busy, lambda r: r.__setitem__(2, 0xFFFFFFFF))),
        ("first-move", corrupt(busy, lambda r: r.__setitem__(2, 0))),  # column 0 is not a red first move
        ("link", corrupt(has_link[0], lambda r: r.__setitem__(P(2, n - 1), 1 << 1))),  # a link starting in the last column
        ("", corrupt(busy, link_without_peg)),
        ("flags", corrupt(busy, lambda r: r.__setitem__(P(6, 1), r[P(6, 1)] | (~(r[P(0, 1)] | r[P(1, 1)]) & 2)))),
    ]
    if rw > 4 + 9 * n:
        cases.append(("padding", corrupt(E - 1, lambda r: r.__setitem__(rw - 1, 1))))
    import torch
    for i, (reason, (bad, e)) in enumerate(cases):
        if np.array_equal(bad, good):
            continue  # the corruption did not apply to this position (e.g. the target bit was already set)
        for device_side in (False, True):
            src = torch.from_numpy(bad.view(np.int32)).to("cuda:0") if device_side else bad
            with pytest.raises(ValueError) as err:
                batch.import_state(src)
            msg = str(err.value)
            assert msg.startswith("invalid state record at index %d:" % e), (i, msg)
            assert reason in msg, (i, reason, msg)
            assert all(np.array_equal(r, init) for r in batch.export_state()), i  # nothing was copied in
    # a sub-range import reports the index within the call's range; the trusted path skips the check
    bad, e = cases[0][1]
    with pytest.raises(ValueError, match=r"^invalid state record at index 0:"):
        batch.import_state(bad[e:e + 1], 7)
    batch.set_validation(False)
    only_counts = good.copy()
    only_counts[busy, 3] += 1  # harmless for the copy itself; never played
    batch.import_state(only_counts)
    assert np.array_equal(batch.export_state(), only_counts)
    batch.set_validation(True)
    batch.close()


def test_clone_gather_checks_device_side_ids():
    """ids on the device are checked by the clone kernel itself (ADVICE r1): a bad id copies nothing for its
    env and fails the call; twixt_clone_from refuses overlapping ranges within one batch."""
    import torch
    from twixt_for_open_spiel_b200 import TwixTBatch
    n, E = 7, 64
    b = TwixTBatch(n, E, 0, SEED)
    b.playout(0, 16, max_plies=9)
    before = b.export_state()
    good = torch.tensor([3, 3, 15, 0], dtype=torch.int64, device="cuda:0")
    b.clone_gather(good, 32)
    after = b.export_state()
    assert np.array_equal(after[32:36], before[[3, 3, 15, 0]])
    for bad_ids in ([3, E, 5, 1], [2, -1, 5, 1], [2, 41, 5, 1]):  # out of range (both sides), inside [40, 44)
        ids = torch.tensor(bad_ids, dtype=torch.int64, device="cuda:0")
        snap = b.export_state()
        with pytest.raises(ValueError, match=r"src_ids\[1\]"):
            b.clone_gather(ids, 40)
        now = b.export_state()
        assert np.array_equal(now[41], snap[41])  # the offending env was not written
        assert np.array_equal(now[40], snap[bad_ids[0]]) and np.array_equal(now[42], snap[5])  # the others were
    with pytest.raises(ValueError, match="overlap"):
        b.clone_from(4, b, 0, 8)
    b.clone_from(32, b, 0, 8)
    assert np.array_equal(b.export_state(32, 8), b.export_state(0, 8))
    b.close()


# ----------------------------------------------------- bounds-instrumented playout kernel ---
def test_playout_kernel_never_leaves_its_envs_storage(tmp_path):
    """compute-sanitizer is closed on this pool, so the playout kernel is built a second time with every
    shared-memory access of the rules and the flood stack, and every blocked-plane reduction, tested against
    the env's own storage (-DTW_PLAYOUT_BOUNDS_CHECK=1).  All 20 board sizes, fresh and mid-game starts with
    swaps: zero violations, and the games still equal the oracle's."""
    from twixt_for_open_spiel_b200 import build
    variant = build.build(out=os.path.join(ROOT, "tests", "_build", "libtwixt_b200_bounds.so"),
                          extra_flags=["-DTW_PLAYOUT_BOUNDS_CHECK=1"])
    code = textwrap.dedent("""
        import sys
        import numpy as np
        sys.path.insert(0, %r)
        from oracle import pyoracle
        from twixt_for_open_spiel_b200 import TwixTBatch
        seed = 0x7477697854
        total = 0
        for n in range(5, 25):
            E = 768
            b = TwixTBatch(n, E, 0, seed)
            b.playout(0, E // 2, max_plies=n)          # half the envs continue from a mid-game position
            rets, lens, _ = b.playout()
            st = b.stats()
            assert st["debug_violations"] == 0, (n, st)
            assert bool(b.is_terminal().all())
            og = pyoracle.OracleGame(n)
            recs = b.export_state()
            for e in list(range(0, E, 37)) + [E // 2 - 1, E // 2, E - 1]:
                s = og.new_initial_state()
                if e < E // 2:
                    s.playout_philox(seed, e, n)
                acts = s.playout_philox(seed, e)
                assert len(acts) == lens[e] and np.array_equal(recs[e], s.export_record()), (n, e)
            total += int(st["plies"])
            b.close()
        print("bounds ok", total)
    """ % ROOT)
    env = dict(os.environ, TWIXT_B200_LIB=variant)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert res.returncode == 0 and "bounds ok" in res.stdout, (res.stdout[-300:], res.stderr[-3000:])


# -------------------------------------------------------------- obs + mask producer ---
@pytest.mark.parametrize("n", [5, 6, 7, 8, 12, 17, 24])
def test_observation_and_mask_producer(oracle_mod, n):
    """BASELINE config C5: [B,12,n,n-2] f32 + [B,n*n] u8 from ONE pass over the records, into torch tensors
    and through DLPack; bit-identical to the separate calls and to the oracle (twixt.cc:101-132, twixt.h:86-90)."""
    import torch
    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.producer import ObservationMaskProducer
    og = oracle_mod.OracleGame(n)
    E = 80
    batch = TwixTBatch(n, E, 0, SEED)
    depth = [(e * 5) % (n * n - 2) for e in range(E)]
    for e in range(E):
        if depth[e]:
            batch.playout(e, 1, max_plies=depth[e], want_returns=False, want_lengths=False)
    prod = ObservationMaskProducer(batch)
    obs, mask = prod.produce()
    assert obs.shape == (E, 12, n, n - 2) and obs.dtype == torch.float32 and obs.is_cuda
    assert mask.shape == (E, n * n) and mask.dtype == torch.uint8
    obs_h, mask_h = obs.cpu().numpy(), mask.cpu().numpy()
    assert np.array_equal(obs_h, batch.observation()) and np.array_equal(mask_h, batch.legal_mask())
    terminal = 0
    for e in range(E):
        s = og.new_initial_state()
        s.playout_philox(SEED, e, depth[e])
        assert np.array_equal(obs_h[e].reshape(-1), s.observation_tensor(0)), (n, e)
        want = np.zeros(n * n, dtype=np.uint8)
        want[s.legal_actions()] = 1
        assert np.array_equal(mask_h[e], want), (n, e)
        terminal += s.is_terminal()
    assert (n > 6) or terminal > 0  # small boards: finished games (all-zero masks) were in the batch
    # DLPack both ways: export capsules, and lend consumer-owned buffers (offset so the mask is not 16-byte aligned)
    cap_obs, cap_mask = prod.produce_dlpack(8, 40)
    o2, m2 = torch.from_dlpack(cap_obs), torch.from_dlpack(cap_mask)
    assert np.array_equal(o2.cpu().numpy(), obs_h[8:48]) and np.array_equal(m2.cpu().numpy(), mask_h[8:48])
    lend_obs = torch.full((E, 12, n, n - 2), -5.0, device="cuda:0")
    lend_raw = torch.full((E * n * n + 3,), 9, dtype=torch.uint8, device="cuda:0")
    o3, m3 = prod.produce(0, E, out_obs=lend_obs.__dlpack__(), out_mask=lend_raw[3:].__dlpack__())
    assert np.array_equal(o3.cpu().numpy(), obs_h) and np.array_equal(m3.cpu().numpy(), mask_h)
    assert (lend_raw[:3] == 9).all()
    # host buffers through the same C entry point
    oh, mh = batch.observation_and_mask(3, 20)
    assert np.array_equal(oh, obs_h[3:23]) and np.array_equal(mh, mask_h[3:23])
    batch.close()


# ---------------------------------------------------------------- device-side replay ---
@pytest.mark.parametrize("n", [5, 8, 12, 24])
def test_replay_whole_histories_in_one_launch(oracle_mod, n):
    """twixt_replay: [B, T] action histories (ragged, with swaps) applied by one launch equal the oracle's
    replay; `lengths` cuts rows; an illegal action stops ITS env there with the reference's message."""
    import torch
    from twixt_for_open_spiel_b200 import SpielFatalError, TwixTBatch
    og = oracle_mod.OracleGame(n)
    rng = random.Random(90 + n)
    B = 64
    games = [random_game_actions(og, rng, force_swap=(i % 3 == 0), max_plies=rng.randrange(0, n * n)) for i in range(B)]
    acts = pad_games(games)
    batch = TwixTBatch(n, B, 0, SEED)
    applied = batch.replay(acts)
    assert applied.tolist() == [len(g) for g in games]
    recs = batch.export_state()
    for e, g in enumerate(games):
        s = og.new_initial_state()
        s.replay(g)
        assert np.array_equal(recs[e], s.export_record()), (n, e)
    # device pointers + explicit lengths (half of every history), continuing with the second halves afterwards
    batch.reset()
    half = np.array([len(g) // 2 for g in games], dtype=np.int32)
    d_acts = torch.from_numpy(acts).to("cuda:0")
    d_applied = torch.zeros(B, dtype=torch.int32, device="cuda:0")
    batch.replay(d_acts, lengths=torch.from_numpy(half).to("cuda:0"), out_applied=d_applied)
    batch.synchronize()
    assert d_applied.cpu().numpy().tolist() == half.tolist()
    rest = pad_games([g[len(g) // 2:] or [-1] for g in games])
    batch.replay(rest)
    assert np.array_equal(batch.export_state(), recs)
    # an illegal action in the middle of env 5's history (its own first move again, two plies later)
    long_env = max(range(B), key=lambda e: len(games[e]))
    assert len(games[long_env]) >= 4
    bad = acts.copy()
    pos = 3
    illegal = int(bad[long_env, 2])  # a cell occupied since ply 2 (pegs are never removed after the swap window)
    bad[long_env, pos] = illegal
    batch.reset()
    with pytest.raises(SpielFatalError, match=r"^Not a legal action: %d$" % illegal):
        batch.replay(bad)
    applied2 = np.zeros(B, dtype=np.int32)
    batch.reset()
    batch.replay(bad, out_applied=applied2, raise_on_illegal=False)
    assert applied2[long_env] == pos and applied2.tolist()[:long_env] == [len(g) for g in games][:long_env]
    s = og.new_initial_state()
    s.replay(games[long_env][:pos])
    assert np.array_equal(batch.export_state(long_env, 1)[0], s.export_record())
    batch.close()


def test_deserialize_uses_device_replay(oracle_mod):
    from twixt_for_open_spiel_b200 import SpielFatalError, load_game
    game = load_game("twixt(board_size=10)")
    og = oracle_mod.OracleGame(10)
    acts = random_game_actions(og, random.Random(4), force_swap=True, max_plies=55)
    st = game.new_initial_state()
    for a in acts:
        st.apply_action(a)
    launches0 = st._pool.stats()["kernel_launches"]
    again = game.deserialize_state(st.serialize())
    assert np.array_equal(again.export_record(), st.export_record()) and again.history() == acts
    if again._pool is st._pool:
        assert again._pool.stats()["kernel_launches"] - launches0 <= 3  # reset + ONE replay launch, not 55 applies
    with pytest.raises(SpielFatalError, match=r"^Not a legal action: %d$" % acts[3]):
        game.deserialize_state("\n".join(str(a) for a in acts[:6] + [acts[3]]))


# ------------------------------------------------------------------ single-state step ---
@pytest.mark.parametrize("n", [5, 8, 13, 24])
def test_step_apply_and_query_in_one_launch(oracle_mod, n):
    """twixt_step: ApplyAction + CurrentPlayer / IsTerminal / Returns / LegalActions of the new state from one
    launch (what the adapters call per move), against the oracle at every ply of games with swaps; reset and
    query modes; an illegal action reports the reference's message and changes nothing."""
    from twixt_for_open_spiel_b200 import SpielFatalError, TwixTBatch
    og = oracle_mod.OracleGame(n)
    rng = random.Random(700 + n)
    batch = TwixTBatch(n, 4, 0, SEED)
    for gi in range(6):
        env = gi % 4
        acts = random_game_actions(og, rng, force_swap=(gi % 2 == 0))
        st = og.new_initial_state()
        launches0 = batch.stats()["kernel_launches"]
        status, player, term, rets, legal = batch.step(env, -2)  # TWIXT_STEP_RESET
        assert (status, player, term, rets) == (0, 0, False, [0.0, 0.0]) and legal.tolist() == st.legal_actions()
        for ply, a in enumerate(acts):
            if ply == 3:  # an occupied cell: illegal, state and answers unchanged
                before = batch.export_state(env, 1)
                with pytest.raises(SpielFatalError, match=r"^Not a legal action: %d$" % acts[2]):
                    batch.step(env, acts[2])
                assert np.array_equal(batch.export_state(env, 1), before)
                _, p2, t2, r2, l2 = batch.step(env, -1)  # TWIXT_STEP_QUERY
                assert (p2, t2, r2, l2.tolist()) == (st.current_player(), st.is_terminal(), st.returns(), st.legal_actions())
            status, player, term, rets, legal = batch.step(env, a)
            st.apply_action(a)
            assert status == 0 and player == st.current_player() and term == st.is_terminal(), (n, gi, ply)
            assert rets == st.returns() and legal.tolist() == st.legal_actions(), (n, gi, ply)
        assert term and player == -4 and len(legal) == 0
        assert np.array_equal(batch.export_state(env, 1)[0], st.export_record())
        assert batch.stats()["kernel_launches"] - launches0 == 1 + len(acts) + 2  # one launch per step, nothing else
    batch.close()
