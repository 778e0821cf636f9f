"""Shared helpers of the test-suite (test infrastructure)."""
import hashlib
import json
import os
import random
from typing import List

import numpy as np

SEED = 0x7477697854  # "twixT"


def random_game_actions(og, rng: random.Random, force_swap: bool = False, max_plies: int = 10**9) -> List[int]:
    """A random legal game on the oracle; optionally answers the first move with the swap."""
    st = og.new_initial_state()
    acts: List[int] = []
    while not st.is_terminal() and len(acts) < max_plies:
        la = st.legal_actions()
        if len(acts) == 1 and force_swap and acts[0] in la:
            a = acts[0]
        else:
            a = rng.choice(la)
        st.apply_action(a)
        acts.append(a)
    return acts


def draw_seeking_actions(og, pattern=(0, 1)) -> List[int]:
    """twixt_test.cc:185-199: alternately LegalActions().at(p0) / .at(p1)."""
    st = og.new_initial_state()
    acts: List[int] = []
    i = 0
    while not st.is_terminal():
        la = st.legal_actions()
        a = la[min(pattern[i % len(pattern)], len(la) - 1)]
        st.apply_action(a)
        acts.append(a)
        i += 1
    return acts


def pad_games(games: List[List[int]], fill: int = -1) -> np.ndarray:
    """[num_games, max_len] int32 action matrix, `fill` past the end of a game."""
    m = max(len(g) for g in games)
    out = np.full((len(games), m), fill, dtype=np.int32)
    for i, g in enumerate(games):
        out[i, :len(g)] = g
    return out


# ---- digests of the reference's outputs (tests/golden/ref_digests.json) --------------------------------------
# A test that compares with the compiled reference feeds the same observables, in the same order, into a Digest
# whichever implementation produced them; the stored digest is what the reference produced on those inputs.
GOLDEN_DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_digests.json")


def golden_digests() -> dict:
    with open(GOLDEN_DIGESTS) as f:
        return json.load(f)


class Digest:
    def __init__(self):
        self.h = hashlib.sha256()

    def add(self, *items) -> "Digest":
        """Integer sequences, float sequences (as float64), arrays (flattened, with their dtype kept by the
        caller), strings, ints, floats and bools; numpy scalars count as the Python value they hold."""
        for it in items:
            if isinstance(it, np.ndarray):
                self.h.update(b"A" + str(it.dtype).encode() + np.ascontiguousarray(it).reshape(-1).tobytes())
            elif isinstance(it, str):
                self.h.update(b"S" + it.encode("utf-8") + b"\0")
            elif isinstance(it, (bool, np.bool_)):
                self.h.update(b"B1" if it else b"B0")
            elif isinstance(it, (list, tuple)):
                self.h.update(b"L" + repr([v.item() if isinstance(v, np.generic) else v for v in it]).encode())
            else:
                self.h.update(b"V" + repr(it.item() if isinstance(it, np.generic) else it).encode())
        return self

    def hex(self) -> str:
        return self.h.hexdigest()
