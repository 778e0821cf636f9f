"""CPU: the position corpus behind test_gpu_multipass.py.  The multi-pass GPU checks compare every env with
these oracle answers, so what the corpus contains is what they provably cover."""
import numpy as np
import pytest

from test_gpu_multipass import CLASSES, KOPEN, SIZES, assignment, corpus


@pytest.mark.parametrize("n", SIZES)
def test_corpus_covers_every_position_class(oracle_mod, n):
    c = corpus(n)
    assert 700 <= c.P <= 1000
    for cl in CLASSES:
        assert any(cl in s for s in c.classes), (n, cl)
    if n == 5:
        assert any("draw_seeking" in s for s in c.classes)
    assert len({r.tobytes() for r in c.records}) == c.P  # distinct states
    for i, cl in enumerate(c.classes):
        rec = c.records[i]
        ply, result, swapped = int(rec[0]), int(rec[1] & 3), bool((rec[1] >> 2) & 1)
        assert ply == len(c.prefixes[i]) and ("swapped" in cl) == swapped, (n, i)
        assert ply <= (3 * n * n) // 5 or result != KOPEN or "draw_seeking" in cl, (n, i)
        assert (result != KOPEN) == bool(c.terminal[i]) == bool({"red_win", "blue_win", "draw"} & cl), (n, i)
        if "ply1_swap_offered" in cl:
            assert ply == 1 and c.mask[i, c.prefixes[i][0]] == 1
    # the answers agree with each other: terminal -> empty list, zero mask, terminal player, +-1 / 0 returns
    term = c.terminal.astype(bool)
    assert (c.counts[term] == 0).all() and (c.mask[term] == 0).all() and (c.player[term] == -4).all()
    assert (c.player[~term] == (c.records[~term, 0] & 1)).all()
    assert np.array_equal(c.returns[:, 0], -c.returns[:, 1])
    assert np.array_equal(c.mask.sum(axis=1), c.counts)
    for i in range(c.P):
        assert np.flatnonzero(c.mask[i]).tolist() == c.legal[i, :c.counts[i]].tolist()
        assert (c.legal[i, c.counts[i]:] == -1).all()


def test_assignment_is_seeded_and_covers_the_corpus():
    a = assignment(768, 30_000, 5)
    assert np.array_equal(a, assignment(768, 30_000, 5)) and not np.array_equal(a, assignment(768, 30_000, 6))
    assert np.array_equal(a[:768], np.arange(768)) and a.min() == 0 and a.max() == 767
    assert np.unique(a[768:]).size == 768  # every position is also gathered
