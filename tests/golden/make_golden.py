#!/usr/bin/env python3
"""Regenerates the committed golden fixtures in this directory FROM THE REFERENCE.

Needs /root/reference (authoring container only):
  * playthrough_n8.json   parsed from the reference's own golden playthrough
        open_spiel/integration_tests/playthroughs/playthrough.txt
        (game constants, 35 actions, the fully dumped states with their legal
        lists, observation tensors, returns) -- and cross-checked here against
        the compiled reference (oracle/_ref) replaying the same actions;
  * ref_games.json        outputs of the compiled, unmodified reference on
        seeded games at n = 5, 6, 8, 12, 24 (random, forced swap, draw-seeking):
        per ply the current player, the CRC32 of the int64 legal list and of the
        float32 observation tensor, plus terminal flag / returns at the end and a
        few complete dumps;
  * ref_strings.json      Board::ToString (twixtboard.cc:278-448) of the compiled reference at EVERY ply of
        the swap, win and draw games of twixt_test.cc and of seeded random games at n = 6, 12, 24 chosen so
        that links of all eight compass directions, both colours, `[swapped]`, `[x has won]`, `[o has won]`
        and `[draw]` occur; with and without ANSI colour codes;
  * kats.json             the known-answer tests of twixt_test.cc restated as data,
        and the Random123 Philox4x32-10 known answers.
The tests never read /root/reference; they read these files.

    python tests/golden/make_golden.py

  * ref_digests.json      (`python tests/golden/make_golden.py digests`, needs no reference tree) SHA-256 digests
        of everything the tests that compare live with the compiled reference check -- the crossing table, the
        seeded random games at every board size, ToString and ActionToString, the CUDA path's lock-step games and
        fused playouts, the golden playthrough -- so those comparisons also run where oracle/_ref is absent.
        Computed with the oracle, the host renderer and the adapter, whose outputs on exactly these inputs those
        same tests found equal to the compiled reference; where oracle/_ref is present the tests still compare
        with it live, so a digest that disagreed with the reference would fail there.
"""
import json
import os
import random
import re
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import pyoracle  # noqa: E402

PLAYTHROUGH = "/root/reference/open_spiel/integration_tests/playthroughs/playthrough.txt"


def crc_list(lst):
    return zlib.crc32(np.asarray(lst, dtype=np.int64).tobytes()) & 0xFFFFFFFF


def crc_obs(obs):
    return zlib.crc32(np.asarray(obs, dtype=np.float32).tobytes()) & 0xFFFFFFFF


def parse_playthrough(path):
    with open(path, encoding="utf-8") as f:
        lines = f.read().split("\n")
    out = {"header": {}, "actions": [], "states": []}
    for ln in lines[:40]:
        m = re.match(r"^(\w+)\(\) = (.*)$", ln)
        if m:
            out["header"][m.group(1)] = m.group(2)
    i = 0
    cur = None
    while i < len(lines):
        ln = lines[i]
        m = re.match(r"^# State (\d+)$", ln)
        if m:
            cur = {"index": int(m.group(1))}
            out["states"].append(cur)
        elif ln.startswith("action: "):
            out["actions"].append(int(ln.split(": ")[1]))
        elif cur is not None:
            if ln.startswith("IsTerminal() = "):
                cur["is_terminal"] = ln.endswith("True")
            elif ln.startswith("History() = "):
                cur["history"] = json.loads(ln.split(" = ", 1)[1])
            elif ln.startswith("CurrentPlayer() = "):
                cur["current_player"] = int(ln.split(" = ")[1])
            elif ln.startswith("Returns() = "):
                cur["returns"] = [float(v) for v in json.loads(ln.split(" = ", 1)[1])]
            elif ln.startswith("LegalActions() = "):
                cur["legal_actions"] = json.loads(ln.split(" = ", 1)[1])
            elif ln.startswith("StringLegalActions() = "):
                cur["string_legal_actions"] = json.loads(ln.split(" = ", 1)[1])
            elif ln.startswith("ObservationString(0) = "):
                cur["observation_string"] = json.loads(ln.split(" = ", 1)[1], strict=False)
            elif re.match(r"^ObservationTensor\((\d)\):$", ln):
                player = int(ln[len("ObservationTensor(")])
                rows = []
                j = i + 1
                while j < len(lines) and lines[j] and lines[j][0] in "◉◯":
                    rows.append(lines[j])
                    j += 1
                n = len(rows)
                planes = [g for g in rows[0].split("  ")]
                w = len(planes[0])
                t = np.zeros((len(planes), n, w), dtype=np.float32)
                for r, row in enumerate(rows):
                    for p, grp in enumerate(row.split("  ")):
                        for c, ch in enumerate(grp):
                            t[p, r, c] = 1.0 if ch == "◉" else 0.0
                cur["obs_shape"] = list(t.shape)
                cur["obs_ones_%d" % player] = np.flatnonzero(t.reshape(-1)).tolist()
                i = j - 1
        i += 1
    return out


def ref_trace(n, actions, full_every=0):
    """Replay on the compiled reference; per-ply digest."""
    rg = pyoracle.RefGame(n)
    st = rg.new_initial_state()
    plies = []
    dumps = {}
    for ply in range(len(actions) + 1):
        la = st.legal_actions()
        obs = st.observation_tensor(0)
        plies.append([st.current_player(), len(la), crc_list(la), crc_obs(obs)])
        if full_every and (ply % full_every == 0 or ply == len(actions)):
            dumps[str(ply)] = {"legal": la, "obs_ones": np.flatnonzero(obs).tolist(),
                               "cells": st.export_cells().reshape(-1).tolist(), "header": st.board_header()[:3]}
        if ply < len(actions):
            st.apply_action(actions[ply])
    res = {"n": n, "actions": list(actions), "plies": plies, "terminal": st.is_terminal(), "returns": st.returns(),
           "dumps": dumps}
    del st
    del rg
    return res


def gen_games():
    from helpers import draw_seeking_actions, random_game_actions
    games = []
    for n, count, full_every in ((5, 12, 1), (6, 6, 4), (8, 8, 9), (12, 4, 30), (24, 3, 150)):
        og = pyoracle.OracleGame(n)
        rng = random.Random(2026 + n)
        for i in range(count):
            acts = random_game_actions(og, rng, force_swap=(i % 2 == 1))
            games.append(ref_trace(n, acts, full_every))
        if n <= 8:
            for pat in ((0, 1), (10**6, 0)):
                games.append(ref_trace(n, draw_seeking_actions(og, pat), full_every))
    return games


def ref_strings(n, actions, ansi):
    rg = pyoracle.RefGame(n, ansi)
    st = rg.new_initial_state()
    all_strings, dirs = [st.to_string()], 0
    for a in actions:
        st.apply_action(a)
        all_strings.append(st.to_string())
    for c in st.export_cells():
        dirs |= int(c[1])
    # the CRC32 of the UTF-8 picture at EVERY ply; the text itself at every ply of a short game, at a few
    # plies (first, last, some in between) of a long one -- keeps the fixture small
    last = len(actions)
    keep = range(last + 1) if last <= 40 else sorted({0, 1, 2, last // 3, 2 * last // 3, last - 1, last})
    res = {"n": n, "ansi": ansi, "actions": list(actions), "strings": {str(k): all_strings[k] for k in keep},
           "crcs": [zlib.crc32(t.encode("utf-8")) & 0xFFFFFFFF for t in all_strings], "link_directions": dirs,
           "returns": st.returns()}
    del st
    del rg
    return res


def gen_strings():
    from helpers import draw_seeking_actions, random_game_actions
    games = []
    og5 = pyoracle.OracleGame(5)
    fixed = [(8, [19, 19, 36]), (8, [21, 38, 15, 11, 27, 17, 42, 45, 48]), (5, draw_seeking_actions(og5, (0, 1)))]
    for n, acts in fixed:
        for ansi in (True, False):
            games.append(ref_strings(n, acts, ansi))
    # seeded random games: keep looking until a red win, a blue win and a swapped game are in the set
    for n, ansi in ((6, True), (12, False), (24, True)):
        og = pyoracle.OracleGame(n)
        rng = random.Random(77 + n)
        want = {"red", "blue", "swap"}
        for i in range(400):
            if not want:
                break
            acts = random_game_actions(og, rng, force_swap=(i % 2 == 1))
            st = og.new_initial_state()
            st.replay(acts)
            tag = "red" if st.returns()[0] > 0 else ("blue" if st.returns()[1] > 0 else None)
            swapped = len(acts) > 1 and acts[0] == acts[1]
            hit = ({tag} if tag else set()) | ({"swap"} if swapped else set())
            if hit & want:
                want -= hit
                games.append(ref_strings(n, acts, ansi))
    all_dirs = 0
    for g in games:
        all_dirs |= g["link_directions"]
    assert all_dirs == 0xFF, all_dirs
    tails = "".join(g["strings"][str(len(g["actions"]))][-24:] for g in games)
    for needle in ("[swapped]", "[x has won]", "[o has won]", "[draw]"):
        assert needle in tails, needle
    return games


def main():
    assert os.path.exists(PLAYTHROUGH), "needs /root/reference"
    pt = parse_playthrough(PLAYTHROUGH)
    # cross-check the parsed golden file against the compiled reference
    rg = pyoracle.RefGame(8)
    st = rg.new_initial_state()
    by_index = {s["index"]: s for s in pt["states"]}
    for ply in range(len(pt["actions"]) + 1):
        s = by_index.get(ply)
        if s is not None and "legal_actions" in s:
            assert st.legal_actions() == s["legal_actions"], ply
            assert np.flatnonzero(st.observation_tensor(0)).tolist() == s["obs_ones_0"], ply
            assert st.current_player() == s["current_player"]
            assert st.to_string() == s["observation_string"], ply
        if ply < len(pt["actions"]):
            st.apply_action(pt["actions"][ply])
    assert st.is_terminal() and st.returns() == [1.0, -1.0]
    del st, rg
    with open(os.path.join(HERE, "playthrough_n8.json"), "w") as f:
        json.dump(pt, f)
    games = gen_games()
    with open(os.path.join(HERE, "ref_games.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_golden.py on oracle/_ref (unmodified reference)", "games": games}, f)
    kats = {
        "swap_n8": {"actions": [19, 19, 36], "source": "twixt_test.cc:108-131"},
        "legal_counts_n8": {"actions": [21, 38, 15, 11, 27, 17, 42, 45, 48],
                            "sizes_before_each": [48, 48, 46, 46, 44, 44, 42, 42, 40], "illegal_at_ply4": 11,
                            "returns": [1.0, -1.0], "source": "twixt_test.cc:133-183"},
        "draw_n5": {"pattern": [0, 1], "returns": [0.0, 0.0], "source": "twixt_test.cc:185-199"},
        "errors": {"30": "board_size out of range [5..24]: 30", "3": "board_size out of range [5..24]: 3",
                   "illegal": "Not a legal action: 11",
                   "bad_param": "Unknown parameter 'bad_param'. Available parameters are: ansi_color_output, board_size",
                   "source": "twixt_test.cc:50-92,156-161"},
        "philox4x32_10": [
            {"ctr": [0, 0, 0, 0], "key": [0, 0], "out": [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]},
            {"ctr": [0xffffffff] * 4, "key": [0xffffffff] * 2, "out": [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]},
            {"ctr": [0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], "key": [0xa4093822, 0x299f31d0],
             "out": [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]},
        ],
    }
    with open(os.path.join(HERE, "kats.json"), "w") as f:
        json.dump(kats, f, indent=1)
    with open(os.path.join(HERE, "ref_strings.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_golden.py on oracle/_ref (unmodified reference)",
                   "games": gen_strings()}, f)
    for name in ("playthrough_n8.json", "ref_games.json", "ref_strings.json", "kats.json"):
        print(name, os.path.getsize(os.path.join(HERE, name)))


def gen_digests():
    import test_gpu_round2
    import test_oracle_vs_reference as ovr
    import test_render
    import ref_gpu_worker
    from twixt_for_open_spiel_b200.render import board_to_string
    from twixt_for_open_spiel_b200.spiel import TwixTState
    from helpers import Digest

    out = {"generator": "tests/golden/make_golden.py digests", "crossing": {}, "random_games": {}, "render": {},
           "action_strings": {}, "cuda_reference": {}}
    for n in (5, 6, 8, 24):
        out["crossing"][str(n)] = ovr.crossing_digest(ovr.oracle_blocker_sets(pyoracle.OracleGame(n), n))
    for n in range(5, 25):
        out["random_games"][str(n)] = ovr.random_games_digest(pyoracle.OracleGame(n), n)
        out["cuda_reference"][str(n)] = ref_gpu_worker.oracle_digests(n, *test_gpu_round2.ref_worker_games(n))
    for n, ansi in test_render.RENDER_CASES:
        out["render"]["%d,%d" % (n, ansi)] = test_render.render_digest(
            pyoracle.OracleGame(n), n, ansi, lambda os_: board_to_string(os_.export_record(), n, ansi))
    for n in test_render.ACTION_STRING_SIZES:

        class _G:
            def board_size(self):
                return n
        fake = TwixTState.__new__(TwixTState)
        fake._game = _G()
        out["action_strings"][str(n)] = Digest().add(
            test_render.action_strings(n, lambda p, a: TwixTState.action_to_string(fake, p, a))).hex()
        fake._game = None
    out["playthrough"] = test_gpu_round2.playthrough_ply_digests(
        pyoracle.OracleGame(8).new_initial_state, lambda st: board_to_string(st.export_record(), 8, True))
    with open(os.path.join(HERE, "ref_digests.json"), "w") as f:
        json.dump(out, f, indent=0)
    print("ref_digests.json", os.path.getsize(os.path.join(HERE, "ref_digests.json")))


if __name__ == "__main__":
    if sys.argv[1:] == ["digests"]:
        gen_digests()
    else:
        main()
