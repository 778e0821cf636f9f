"""The fused playout kernel's border-flag flood with a set of columns as its work list
(flood_visit_columns in csrc/twixt_engine.cuh), checked on the CPU: tests/flood_columns_harness.cc runs the
kernel's loop on its 8n + 4-word shared-memory layout, pad words poisoned, and must reproduce the oracle's
actions and final record at every board size -- fresh games, swap games and games taken over mid-game --
while taking no more flood visits than the entry stack it replaces."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "twixt_for_open_spiel_b200", "csrc")
SEED = 0x7477697854


@pytest.fixture(scope="module")
def fc():
    out_dir = os.path.join(HERE, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libfloodcolumns.so")
    src = os.path.join(HERE, "flood_columns_harness.cc")
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-fPIC", "-shared", "-I", CSRC, "-o", so, src])
    lib = C.CDLL(so)
    lib.fc_playout.restype = C.c_int
    lib.fc_playout.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return lib


def P(a):
    return a.ctypes.data_as(C.c_void_p)


def _start(og, n, s):
    """the record and oracle state a game starts from: fresh, or taken over mid-game (s % 3 == 2; at ply 1,
    before a possible swap, when s % 6 == 5)"""
    st = og.new_initial_state()
    if s % 3 == 2:
        st.playout_philox(7, s, 1 if s % 6 == 5 else 2 + s % 40)  # plays the state forward
    return st.export_record().astype(np.uint32).copy(), st


@pytest.mark.parametrize("n", list(range(5, 25)))
def test_column_flood_matches_oracle(fc, oracle_mod, n):
    og = oracle_mod.OracleGame(n)
    visits = {0: C.c_int64(0), 1: C.c_int64(0)}
    swaps = 0
    for s in range(120 if n <= 6 else 24):
        stream = s + (n << 33)
        for columns in (1, 0):
            rec, st = _start(og, n, s)
            acts = np.zeros(n * n, dtype=np.int64)
            L = fc.fc_playout(P(rec), n, SEED, stream, 1 << 30, columns, P(acts), C.byref(visits[columns]))
            assert acts[:L].tolist() == st.playout_philox(SEED, stream), (n, s, columns)
            assert np.array_equal(rec, st.export_record()), (n, s, columns)
            if columns:
                swaps += int(rec[1] >> 2) & 1
    assert visits[1].value <= visits[0].value, (visits[1].value, visits[0].value)
    if n <= 6:
        assert swaps >= 3  # the swap path was really taken


@pytest.mark.parametrize("n", [8, 24])
def test_column_flood_stops_at_max_plies(fc, oracle_mod, n):
    og = oracle_mod.OracleGame(n)
    for s in range(12):
        rec, st = _start(og, n, s)
        acts = np.zeros(n * n, dtype=np.int64)
        v = C.c_int64(0)
        L = fc.fc_playout(P(rec), n, SEED, s, 5 + 7 * s, 1, P(acts), C.byref(v))
        assert acts[:L].tolist() == st.playout_philox(SEED, s, 5 + 7 * s)
        assert np.array_equal(rec, st.export_record())
