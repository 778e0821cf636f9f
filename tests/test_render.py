"""ToString parity (SURVEY 8f row 1): the host renderer over an exported record reproduces the reference's
board picture byte for byte -- against the golden playthrough strings, stored digests of the reference's pictures
and, where it is present, the compiled reference itself."""
import json
import os
import random

import pytest

from helpers import Digest, golden_digests, random_game_actions

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_playthrough_strings(oracle_mod):
    from twixt_for_open_spiel_b200.render import board_to_string
    with open(os.path.join(GOLDEN, "playthrough_n8.json")) as f:
        pt = json.load(f)
    st = oracle_mod.OracleGame(8).new_initial_state()
    by_index = {s["index"]: s for s in pt["states"]}
    checked = 0
    for ply in range(36):
        s = by_index.get(ply)
        if s is not None and "observation_string" in s:
            assert board_to_string(st.export_record(), 8, True) == s["observation_string"], ply
            checked += 1
        if ply < 35:
            st.apply_action(pt["actions"][ply])
    assert checked >= 9
    assert board_to_string(st.export_record(), 8, True).endswith("[x has won]")


RENDER_CASES = [(5, True), (6, False), (8, True), (11, False), (12, True), (24, True), (24, False)]
ACTION_STRING_SIZES = (5, 8, 12, 24)


def render_digest(og, n, ansi, to_string):
    """ToString every 4 plies and at the end of seeded random games (forced swap in every other one);
    `to_string(oracle_state)` gives the picture to digest."""
    rng = random.Random(n)
    dg = Digest()
    for gi in range(6 if n <= 12 else 2):
        acts = random_game_actions(og, rng, force_swap=(gi % 2 == 0))
        os_ = og.new_initial_state()
        for ply, a in enumerate(acts):
            if ply % 4 == 0:
                dg.add(to_string(os_))
            os_.apply_action(a)
        dg.add(to_string(os_))
    return dg.hex()


@pytest.mark.parametrize("n,ansi", RENDER_CASES)
def test_matches_compiled_reference(oracle_mod, have_ref, n, ansi):
    """The host renderer against the stored digest of the reference's ToString on these games
    (tests/golden/ref_digests.json), and against the compiled reference itself where it is present."""
    from twixt_for_open_spiel_b200.render import board_to_string
    og = oracle_mod.OracleGame(n)
    got = render_digest(og, n, ansi, lambda os_: board_to_string(os_.export_record(), n, ansi))
    assert got == golden_digests()["render"]["%d,%d" % (n, ansi)]
    if not have_ref:
        return
    rg = oracle_mod.RefGame(n, ansi)
    proto = rg.new_initial_state()
    rng = random.Random(n)
    for gi in range(6 if n <= 12 else 2):
        acts = random_game_actions(og, rng, force_swap=(gi % 2 == 0))
        rs, os_ = proto.clone(), og.new_initial_state()
        for ply, a in enumerate(acts):
            if ply % 4 == 0:
                assert board_to_string(os_.export_record(), n, ansi) == rs.to_string(), (n, gi, ply)
            rs.apply_action(a)
            os_.apply_action(a)
        assert board_to_string(os_.export_record(), n, ansi) == rs.to_string()
        del rs
    del proto, rg


def action_strings(n, action_to_string):
    return [action_to_string(p, a) for a in range(n * n) for p in (0, 1)]


def test_action_to_string_matches_reference(oracle_mod, have_ref):
    """twixt.cc:67-74; also pinned by StringLegalActions in the playthrough (GPU test).  Against the stored
    digest of the reference's strings (tests/golden/ref_digests.json) and the compiled reference where present."""
    from twixt_for_open_spiel_b200.spiel import TwixTState
    want = golden_digests()["action_strings"]
    for n in ACTION_STRING_SIZES:

        class _G:
            def board_size(self):
                return n
        fake = TwixTState.__new__(TwixTState)
        fake._game = _G()
        ours = action_strings(n, lambda p, a: TwixTState.action_to_string(fake, p, a))
        fake._game = None
        assert Digest().add(ours).hex() == want[str(n)], n
        if have_ref:
            rg = oracle_mod.RefGame(n)
            rs = rg.new_initial_state()
            assert ours == action_strings(n, rs.action_to_string), n
            del rs, rg


def test_reference_generated_strings(oracle_mod):
    """tests/golden/ref_strings.json (the compiled reference's ToString at every ply of swap / win / draw and
    random games, all eight link directions, ANSI on and off) against the host renderer over oracle records."""
    import zlib
    from twixt_for_open_spiel_b200.render import board_to_string
    with open(os.path.join(GOLDEN, "ref_strings.json")) as f:
        games = json.load(f)["games"]
    dirs = 0
    for g in games:
        st = oracle_mod.OracleGame(g["n"]).new_initial_state()
        for ply in range(len(g["actions"]) + 1):
            text = board_to_string(st.export_record(), g["n"], g["ansi"])
            assert zlib.crc32(text.encode("utf-8")) & 0xFFFFFFFF == g["crcs"][ply], (g["n"], ply)
            if str(ply) in g["strings"]:
                assert text == g["strings"][str(ply)]
            if ply < len(g["actions"]):
                st.apply_action(g["actions"][ply])
        dirs |= g["link_directions"]
    assert dirs == 0xFF
