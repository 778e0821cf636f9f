"""Pins the oracle (oracle/twixt_oracle.c) BEFORE it is trusted as the checker:

1. against the reference's own known-answer tests (twixt_test.cc) and its golden
   playthrough (playthrough.txt), both restated as committed fixtures;
2. against the unmodified reference compiled into oracle/_ref, move by move, on
   seeded random games at every board size -- and, whether or not oracle/_ref is
   present, against digests of what the reference produced on the same inputs
   (tests/golden/ref_digests.json).
"""
import json
import os
import random
import zlib

import numpy as np
import pytest

from helpers import Digest, draw_seeking_actions, golden_digests, random_game_actions

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def _impls(oracle_mod, have_ref):
    impls = [("oracle", oracle_mod.OracleGame)]
    if have_ref:
        impls.append(("reference", oracle_mod.RefGame))
    return impls


def test_reference_is_available_here(have_ref):
    """In the authoring container the reference must compile (DESIGN.md: oracle is PINNED)."""
    if os.path.isdir("/root/reference"):
        assert have_ref


def test_philox_known_answers(oracle_mod):
    for kat in _load("kats.json")["philox4x32_10"]:
        assert oracle_mod.philox(kat["ctr"], kat["key"]) == kat["out"]


def test_parameter_errors(oracle_mod, have_ref):
    """twixt_test.cc:50-92."""
    errs = _load("kats.json")["errors"]
    for name, Game in _impls(oracle_mod, have_ref):
        Game(10)
        for bad in (30, 3):
            with pytest.raises(oracle_mod.SpielError) as e:
                Game(bad)
            assert str(e.value) == errs[str(bad)], name
    if have_ref:
        import ctypes as C
        buf = C.create_string_buffer(256)
        assert oracle_mod.ref_lib().ref_game_new_with_param(b"bad_param", 3, buf, 256) == 1
        assert buf.value.decode() == errs["bad_param"]


def test_swap_kat(oracle_mod, have_ref):
    """twixt_test.cc:108-131."""
    for name, Game in _impls(oracle_mod, have_ref):
        st = Game(8).new_initial_state()
        assert st.current_player() == 0 and 11 in st.legal_actions()
        st.apply_action(19)
        assert st.current_player() == 1
        st.apply_action(19)
        la = st.legal_actions()
        assert 19 in la and 29 not in la and len(la) == 47 and st.current_player() == 0
        st.apply_action(36)
        la = st.legal_actions()
        assert 19 in la and 29 not in la and 36 not in la and len(la) == 46
        del st


def test_legal_counts_and_win_kat(oracle_mod, have_ref):
    """twixt_test.cc:133-183."""
    kat = _load("kats.json")["legal_counts_n8"]
    for name, Game in _impls(oracle_mod, have_ref):
        st = Game(8).new_initial_state()
        for ply, (a, size) in enumerate(zip(kat["actions"], kat["sizes_before_each"])):
            assert len(st.legal_actions()) == size, (name, ply)
            if ply == 4:
                with pytest.raises(oracle_mod.SpielError) as e:
                    st.apply_action(kat["illegal_at_ply4"])
                assert str(e.value) == "Not a legal action: 11"
                assert len(st.legal_actions()) == size
            st.apply_action(a)
        assert st.is_terminal() and st.returns() == kat["returns"] and st.current_player() == -4
        assert st.legal_actions() == []
        del st


def test_draw_kat(oracle_mod, have_ref):
    """twixt_test.cc:185-199."""
    for name, Game in _impls(oracle_mod, have_ref):
        g = Game(5)
        acts = draw_seeking_actions(g, (0, 1))
        assert acts == [5, 2, 6, 3, 7, 8, 9, 11, 10, 12, 13, 16, 14, 17, 15, 18, 19, 21]
        st = g.new_initial_state()
        st.replay(acts)
        assert st.is_terminal() and st.returns() == [0.0, 0.0]
        del st, g


def test_golden_playthrough(oracle_mod, have_ref):
    """open_spiel/integration_tests/playthroughs/playthrough.txt (n=8, 35 moves, red wins)."""
    pt = _load("playthrough_n8.json")
    assert pt["header"]["NumDistinctActions"] == "64" and pt["header"]["MaxGameLength"] == "61"
    assert pt["header"]["ObservationTensorShape"] == "[12, 8, 6]"
    assert len(pt["actions"]) == 35
    by_index = {s["index"]: s for s in pt["states"]}
    dumped = [i for i, s in by_index.items() if "legal_actions" in s]
    assert set(dumped) >= {0, 1, 2, 3, 4, 5, 20, 21}
    for name, Game in _impls(oracle_mod, have_ref):
        g = Game(8)
        assert g.num_distinct_actions() == 64 and g.max_game_length() == 61
        st = g.new_initial_state()
        for ply in range(36):
            s = by_index.get(ply)
            if s is not None and "current_player" in s:
                assert st.current_player() == s["current_player"], (name, ply)
                assert st.is_terminal() == s["is_terminal"]
                assert st.returns() == s["returns"]
                if "legal_actions" in s:
                    assert st.legal_actions() == s["legal_actions"], (name, ply)
                for p in (0, 1):  # the tensor ignores the player argument
                    if "obs_ones_%d" % p in s:
                        assert np.flatnonzero(st.observation_tensor(p)).tolist() == s["obs_ones_%d" % p], (name, ply)
            if ply < 35:
                st.apply_action(pt["actions"][ply])
        assert st.is_terminal() and st.current_player() == -4 and st.returns() == [1.0, -1.0]
        del st, g


DX = [1, 2, 2, 1, -1, -2, -2, -1]
DY = [2, 1, -1, -2, -2, -1, 1, 2]


def oracle_blocker_sets(og, n):
    """{(x, y, d): the links that block link (x, y, d)}, each blocker named from both of its ends as the
    reference's BlockerMap holds it."""
    out = {}
    for x in range(n):
        for y in range(n):
            for d in range(8):
                both = set()
                for bx, by, bd in og.blockers(x, y, d):
                    both.add((bx, by, bd))
                    both.add((bx + DX[bd], by + DY[bd], (bd + 4) % 8))
                out[(x, y, d)] = both
    return out


def crossing_digest(sets):
    dg = Digest()
    for key in sorted(sets):
        dg.add(list(key), sorted(sets[key]))
    return {"entries": sum(len(v) for v in sets.values()), "digest": dg.hex()}


def test_crossing_relation_equals_reference_table(oracle_mod, have_ref):
    """The geometric blocker relation == BlockerMap built from kLinkDescriptorTable
    (twixtboard.cc:38-144, 176-190), link by link; entry totals as in SURVEY 8(a).  Against the compiled
    reference where it is present, and always against the reference's stored table (tests/golden/ref_digests.json)."""
    want = golden_digests()["crossing"]
    for n, want_entries in ((5, 992), (6, None), (8, 4928), (24, 69696)):
        og = oracle_mod.OracleGame(n)
        sets = oracle_blocker_sets(og, n)
        assert crossing_digest(sets) == want[str(n)], n
        if want_entries is not None:
            assert want[str(n)]["entries"] == want_entries
        if have_ref:
            rg = oracle_mod.RefGame(n)
            keep = rg.new_initial_state()  # builds the process-global map for this size
            for (x, y, d), both in sets.items():
                assert set(rg.blockers(x, y, d)) == both, (n, x, y, d)
            del keep, rg


def random_games_digest(game, n):
    """Seeded random games (forced swap in 1/3) on `game`, every observable the live comparison below checks, in
    its order, and five Philox playouts."""
    proto = game.new_initial_state()
    rng = random.Random(n)
    dg = Digest()
    for gi in range(20 if n <= 12 else 6):
        st = proto.clone()
        ply, first = 0, None
        while True:
            la = st.legal_actions()
            dg.add(la, st.current_player(), st.is_terminal(), st.returns())
            if ply % 6 == 0 or st.is_terminal():
                dg.add(st.observation_tensor(0), st.export_cells(), st.board_header()[:3],
                       st.legal_list_of(0), st.legal_list_of(1))
            if st.is_terminal():
                break
            a = first if (ply == 1 and gi % 3 == 0 and first in la) else rng.choice(la)
            if ply == 0:
                first = a
            st.apply_action(a)
            ply += 1
        del st
    for s in range(5):
        dg.add(proto.clone().playout_philox(99, s))
    del proto
    return dg.hex()


@pytest.mark.parametrize("n", list(range(5, 25)))
def test_oracle_equals_reference_on_random_games(oracle_mod, have_ref, n):
    """Move by move against the compiled reference where it is present; always against the digest of what the
    reference produced on the same games (tests/golden/ref_digests.json)."""
    assert random_games_digest(oracle_mod.OracleGame(n), n) == golden_digests()["random_games"][str(n)]
    if not have_ref:
        return
    rg = oracle_mod.RefGame(n)
    og = oracle_mod.OracleGame(n)
    proto = rg.new_initial_state()
    rng = random.Random(n)
    for gi in range(20 if n <= 12 else 6):
        rs, os_ = proto.clone(), og.new_initial_state()
        ply, first = 0, None
        while True:
            la = rs.legal_actions()
            assert la == os_.legal_actions(), (n, gi, ply)
            assert rs.current_player() == os_.current_player()
            assert rs.is_terminal() == os_.is_terminal() and rs.returns() == os_.returns()
            if ply % 6 == 0 or rs.is_terminal():
                assert np.array_equal(rs.observation_tensor(0), os_.observation_tensor(1))
                assert np.array_equal(rs.export_cells(), os_.export_cells()), (n, gi, ply)
                assert rs.board_header()[:3] == os_.board_header()[:3]
                for p in (0, 1):
                    assert rs.legal_list_of(p) == os_.legal_list_of(p)
            if rs.is_terminal():
                break
            a = first if (ply == 1 and gi % 3 == 0 and first in la) else rng.choice(la)
            if ply == 0:
                first = a
            rs.apply_action(a)
            os_.apply_action(a)
            ply += 1
        del rs
    # the Philox policy restated on both sides plays identical games
    for s in range(5):
        rs, os_ = proto.clone(), og.new_initial_state()
        assert rs.playout_philox(99, s) == os_.playout_philox(99, s)
        del rs
    del proto, rg


def test_oracle_matches_reference_generated_fixture(oracle_mod):
    """tests/golden/ref_games.json: outputs of the unmodified reference, committed."""
    data = _load("ref_games.json")
    assert len(data["games"]) >= 30
    for g in data["games"]:
        og = oracle_mod.OracleGame(g["n"])
        st = og.new_initial_state()
        for ply, (player, count, crc_l, crc_o) in enumerate(g["plies"]):
            la = st.legal_actions()
            assert st.current_player() == player and len(la) == count
            assert (zlib.crc32(np.asarray(la, dtype=np.int64).tobytes()) & 0xFFFFFFFF) == crc_l
            obs = st.observation_tensor(0)
            assert (zlib.crc32(obs.tobytes()) & 0xFFFFFFFF) == crc_o
            d = g["dumps"].get(str(ply))
            if d is not None:
                assert la == d["legal"] and np.flatnonzero(obs).tolist() == d["obs_ones"]
                assert st.export_cells().reshape(-1).tolist() == d["cells"]
                assert st.board_header()[:3] == d["header"]
            if ply < len(g["actions"]):
                st.apply_action(g["actions"][ply])
        assert st.is_terminal() == g["terminal"] and st.returns() == g["returns"]


def test_fixture_generator_is_reproducible(oracle_mod, have_ref):
    """Where /root/reference exists, re-parse its playthrough and compare with the committed file."""
    path = "/root/reference/open_spiel/integration_tests/playthroughs/playthrough.txt"
    if not os.path.exists(path):
        pytest.skip("reference tree not present (GPU box)")
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLDEN, "make_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert json.loads(json.dumps(mod.parse_playthrough(path))) == _load("playthrough_n8.json")
