"""The blocked-neighbour plane derived from the position (derive_blocked_word, csrc/twixt_engine.cuh) against
the per-move rule that the apply kernel, the host engine and the oracle keep.  The fused playout kernel no longer
writes the plane move by move; derive_blocked_kernel ORs in the bits of the knight pairs a launch formed.

CPU: tests/blocked_harness.cc compiles the derivation for the host next to host_engine_harness.cc.
GPU (-m gpu): the exported records after twixt_playout, bit for bit, at every board size, from fresh,
mid-game and hand-made starting records."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from helpers import SEED, random_game_actions

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "twixt_for_open_spiel_b200", "csrc")
P_RED, P_BLUE, P_LINK0, P_BLOCKED, HDR = 0, 1, 2, 8, 4
# east knight offsets of the link planes P_LINK0 + 0..3: NNE, ENE, ESE, SSE
EAST = ((1, 2), (2, 1), (2, -1), (1, -2))


@pytest.fixture(scope="module")
def bh():
    out_dir = os.path.join(HERE, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libblockedharness.so")
    srcs = [os.path.join(HERE, "blocked_harness.cc"), os.path.join(HERE, "host_engine_harness.cc")] + \
        [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-x", "c++", "-fPIC", "-shared", "-I", CSRC,
                               "-I", HERE, "-o", so, os.path.join(HERE, "blocked_harness.cc")])
    lib = C.CDLL(so)
    lib.he_init.argtypes = [C.c_void_p, C.c_int]
    lib.he_apply.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.bh_derive_blocked.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    for fn in (lib.he_playout, lib.bh_playout_derived):
        fn.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p]
    return lib


def P(a):
    return a.ctypes.data_as(C.c_void_p)


def plane(rec, n, p):
    return rec[HDR + p * n: HDR + (p + 1) * n]


def derived(bh, rec, n):
    out = np.zeros(n, dtype=np.uint32)
    bh.bh_derive_blocked(P(rec), n, P(out))
    return out


def midgame_record(oracle_mod, n, rng, plies, force_swap=False):
    og = oracle_mod.OracleGame(n)
    st = og.new_initial_state()
    st.replay(random_game_actions(og, rng, force_swap=force_swap, max_plies=plies))
    return st.export_record().astype(np.uint32)


def unblock_a_pair(rec, n):
    """Hand-made record: clear the blocked bit of one refused knight pair, leaving the two pegs unlinked and
    unblocked -- a record the import validator accepts (blocked bits only have to sit on pegs) but no game
    reaches.  Returns the cell, or None if the position has no blocked pair."""
    pegs = (plane(rec, n, P_RED), plane(rec, n, P_BLUE))
    blk = plane(rec, n, P_BLOCKED)
    for x in range(n):
        for y in range(n):
            if not (blk[x] >> y) & 1:
                continue
            for c in pegs:
                if (c[x] >> y) & 1:
                    for d, (dx, dy) in enumerate(EAST):
                        tx, ty = x + dx, y + dy
                        if tx < n and 0 <= ty < n and (c[tx] >> ty) & 1 and not (plane(rec, n, P_LINK0 + d)[x] >> y) & 1:
                            rec[HDR + P_BLOCKED * n + x] &= np.uint32(~(1 << y) & 0xFFFFFFFF)
                            return x, y
    return None


@pytest.mark.parametrize("n", [5, 6, 8, 11, 12, 17, 24])
def test_derived_plane_equals_per_move_plane_after_every_ply(bh, oracle_mod, n):
    og = oracle_mod.OracleGame(n)
    rng = random.Random(1000 + n)
    R = og.record_words()
    blocked_seen = 0
    for g in range(12 if n <= 12 else 6):
        rec = np.zeros(R, dtype=np.uint32)
        bh.he_init(P(rec), n)
        st = og.new_initial_state()
        for a in random_game_actions(og, rng, force_swap=(g % 3 == 0)):
            assert bh.he_apply(P(rec), n, a) == 0
            st.apply_action(a)
            assert np.array_equal(rec, st.export_record())
            assert np.array_equal(derived(bh, rec, n), plane(rec, n, P_BLOCKED)), (n, g, a)
        blocked_seen += int(plane(rec, n, P_BLOCKED).any())
    assert blocked_seen > 0  # the games did refuse links


@pytest.mark.parametrize("n", [5, 7, 8, 12, 16, 20, 24])
def test_playout_with_derivation_matches_per_move_rule(bh, oracle_mod, n):
    """Fresh, ply-1 (before a possible swap) and mid-game starts: the kernel-structured playout without blocked
    bookkeeping plus the derivation pass ends in the same record as the per-move rule."""
    rng = random.Random(2000 + n)
    R = oracle_mod.OracleGame(n).record_words()
    for s in range(18):
        plies = (0, 1, rng.randrange(2, n * n // 2))[s % 3]
        start = midgame_record(oracle_mod, n, rng, plies, force_swap=(s % 6 == 4))
        assert len(start) == R
        a, b = start.copy(), start.copy()
        acts_a, acts_b = np.zeros(n * n, dtype=np.int64), np.zeros(n * n, dtype=np.int64)
        la = bh.he_playout(P(a), n, SEED, s, 1 << 30, P(acts_a))
        lb = bh.bh_playout_derived(P(b), n, SEED, s, 1 << 30, P(acts_b))
        assert la == lb and np.array_equal(acts_a[:la], acts_b[:lb])
        assert np.array_equal(a, b), (n, s, plies)


@pytest.mark.parametrize("n", [6, 9, 12, 18, 24])
def test_handmade_unblocked_pair_plays_out_as_per_move_rule(bh, oracle_mod, n):
    """A validator-accepted record with an unlinked, unblocked knight pair: the per-move rule never examines
    that pair, so its bit stays clear; the derivation only counts pairs with a peg placed during the playout."""
    rng = random.Random(3000 + n)
    made = 0
    for s in range(40):
        rec = midgame_record(oracle_mod, n, rng, rng.randrange(n, n * n // 2))
        cell = unblock_a_pair(rec, n)
        if cell is None:
            continue
        made += 1
        x, y = cell
        assert ((derived(bh, rec, n)[x] >> y) & 1) == 1  # a derivation over the whole board would set it
        a, b = rec.copy(), rec.copy()
        bh.he_playout(P(a), n, SEED, 77 + s, 1 << 30, None)
        bh.bh_playout_derived(P(b), n, SEED, 77 + s, 1 << 30, None)
        assert np.array_equal(a, b), (n, s, cell)
    assert made >= 3


# ---------------------------------------------------------------------------------------------- GPU ---

def _device_playout(n, starts, ids):
    from twixt_for_open_spiel_b200 import TwixTBatch
    b = TwixTBatch(n, len(starts), 0, SEED)
    b.import_state(np.stack(starts))  # validated
    rets, lens, _ = b.playout(stream_ids=ids)
    recs = b.export_state()
    b.close()
    return recs, lens


@pytest.mark.gpu
@pytest.mark.parametrize("n", list(range(5, 25)))
def test_gpu_playout_records_fresh_and_midgame(oracle_mod, n):
    """Every board size: records after twixt_playout equal the oracle's (blocked plane included) from fresh,
    ply-1 and mid-game starting records in one launch."""
    og = oracle_mod.OracleGame(n)
    rng = random.Random(4000 + n)
    starts, states = [], []
    for i in range(48):
        plies = (0, 1, rng.randrange(2, n * n // 2))[i % 3]
        st = og.new_initial_state()
        st.replay(random_game_actions(og, rng, force_swap=(i % 6 == 4), max_plies=plies))
        starts.append(st.export_record().astype(np.uint32))
        states.append(st)
    ids = np.arange(len(starts), dtype=np.uint64) * np.uint64(31) + np.uint64(n)
    recs, lens = _device_playout(n, starts, ids)
    for i, st in enumerate(states):
        oa = st.playout_philox(SEED, int(ids[i]))
        assert lens[i] == len(oa)
        assert np.array_equal(recs[i], st.export_record()), (n, i)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [6, 9, 12, 18, 24])
def test_gpu_handmade_unblocked_pair(bh, oracle_mod, n):
    """Hand-made records through the validated import: the device playout ends in the per-move rule's record."""
    rng = random.Random(5000 + n)
    starts = []
    while len(starts) < 24:
        rec = midgame_record(oracle_mod, n, rng, rng.randrange(n, n * n // 2))
        if unblock_a_pair(rec, n) is not None:
            starts.append(rec)
    ids = np.arange(len(starts), dtype=np.uint64) + np.uint64(900)
    recs, _ = _device_playout(n, starts, ids)
    for i, rec in enumerate(starts):
        want = rec.copy()
        bh.he_playout(P(want), n, SEED, int(ids[i]), 1 << 30, None)
        assert np.array_equal(recs[i], want), (n, i)
