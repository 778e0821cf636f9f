"""-m gpu: the persistent kernels past their first resident wave.

Every persistent kernel handles one env, then moves on to the next one of the range: the legal-list and mask
kernels prefetch the next env's inputs and reuse their staged shared-memory row, the observation kernel
prefetches the next record and reuses its double-buffered bulk-store tile, validation and reset / clone stride
over the range, and a lane of the fused playout kernel that has finished its game takes the next env by
ticket with whatever per-lane state the last game left.  The other tests compare these kernels with the
oracle at a few hundred envs, i.e. within one resident wave; here they run at counts chosen from the
hardware's resident bound (at least three passes) and EVERY env of every call is compared.

The inputs are a corpus of ~768 oracle positions per board size (`corpus`): ply 0, ply 1 with the swap
offered, swapped, early, mid and near-full positions, red wins, blue wins and draws, and at n = 5 the
draw-seeking games.  A batch is filled by importing the corpus into envs [0, P) and gathering [P, E) from a
seeded random assignment, so the expected outputs are the corpus answers gathered by the same assignment; an
env that read its neighbour's or a stride-away env's data would see another position.

The CPU-only checks of the corpus itself are in test_multipass_corpus.py.
"""
import functools
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import SEED, draw_seeking_actions, random_game_actions

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SIZES = list(range(5, 25))
CORPUS_POSITIONS = 768
# position classes the corpus must contain at every board size (test_multipass_corpus.py)
CLASSES = ("ply0", "ply1_swap_offered", "swapped", "early", "mid", "near_full", "red_win", "blue_win", "draw")
KOPEN, KRED, KBLUE, KDRAW = 0, 1, 2, 3  # the result field of a record's header word 1 (twixt_engine.cuh)


# ------------------------------------------------------------------------------------ the corpus ---
class Corpus:
    """P oracle positions of one board size with everything the API kernels answer about them."""

    def __init__(self, n, prefixes, classes, og):
        self.n, self.og = n, og
        self.prefixes = prefixes  # action history of each position
        self.classes = classes    # set of CLASSES (and "draw_seeking") per position
        self.P = P = len(prefixes)
        m = n * (n - 2)
        self.records = np.zeros((P, og.record_words()), dtype=np.uint32)
        self.legal = np.full((P, m), -1, dtype=np.int64)  # ascending list, -1 past the count
        self.counts = np.zeros(P, dtype=np.int32)
        self.mask = np.zeros((P, n * n), dtype=np.uint8)
        self.obs = np.zeros((P, 12 * n * (n - 2)), dtype=np.float32)
        self.player = np.zeros(P, dtype=np.int8)
        self.terminal = np.zeros(P, dtype=np.uint8)
        self.returns = np.zeros((P, 2), dtype=np.float32)
        for i, pre in enumerate(prefixes):
            st = self.state(i)
            la = st.legal_actions()
            self.records[i] = st.export_record()
            self.legal[i, :len(la)] = la
            self.counts[i] = len(la)
            self.mask[i, la] = 1
            self.obs[i] = st.observation_tensor(0)
            self.player[i] = st.current_player()
            self.terminal[i] = st.is_terminal()
            self.returns[i] = st.returns()

    def state(self, i):
        st = self.og.new_initial_state()
        assert st.replay(self.prefixes[i]) == len(self.prefixes[i])
        return st


def _classify(n, acts, ply, og):
    """Classes of the position after acts[:ply] of a complete game `acts`."""
    out = set()
    if ply == 0:
        return {"ply0"}
    swapped = ply >= 2 and acts[1] == acts[0]
    if swapped:
        out.add("swapped")
    if ply == len(acts):  # the game's end
        st = og.new_initial_state()
        st.replay(acts)
        r = st.returns()
        out.add("red_win" if r[0] > 0 else ("blue_win" if r[1] > 0 else "draw"))
        return out
    cells = n * n
    if ply == 1:
        st = og.new_initial_state()
        st.apply_action(acts[0])
        if acts[0] in st.legal_actions():
            out.add("ply1_swap_offered")
    elif ply < cells // 5:
        out.add("early")
    elif ply < (2 * cells) // 5:
        out.add("mid")
    else:
        out.add("near_full")
    return out


@functools.lru_cache(maxsize=None)
def corpus(n, P=CORPUS_POSITIONS):
    """~P distinct positions from seeded random games (a third with a forced swap), cut at chosen plies; games
    are added until every class of CLASSES is present (bounded)."""
    from oracle import pyoracle
    og = pyoracle.OracleGame(n)
    rng = random.Random(SEED + 7919 * n)
    seen, prefixes, classes = set(), [], []

    def add(acts, ply, extra=()):
        st = og.new_initial_state()
        st.replay(acts[:ply])
        key = st.export_record().tobytes()  # distinct states, not just distinct histories
        if key in seen:
            return
        seen.add(key)
        prefixes.append(list(acts[:ply]))
        classes.append(_classify(n, acts, ply, og) | set(extra))

    add([], 0)
    if n == 5:  # twixt_test.cc:185-199 and variations: long games that end in draws
        for pat in [(0, 1), (0, 0), (10**6, 10**6), (1, 0), (2, 3), (0, 10**6)]:
            g = draw_seeking_actions(og, pat)
            for ply in sorted({1, 2, len(g) // 2, len(g) - 2, len(g)}):
                add(g, ply, ("draw_seeking",))
    near_full = (3 * n * n) // 5
    games = 0
    while (len(prefixes) < P or not all(any(c in cl for cl in classes) for c in CLASSES)) and games < 4 * P:
        g = random_game_actions(og, rng, force_swap=(games % 3 == 0))
        games += 1
        L = len(g)
        cuts = {L, 1} if games % 2 == 0 else {L}
        hi = min(L - 1, near_full)
        if hi >= 2:
            cuts |= {rng.randint(2, hi) for _ in range(6)}
            cuts.add(rng.randint(max(2, (2 * n * n) // 5), hi) if hi >= (2 * n * n) // 5 else hi)
        for ply in sorted(cuts):
            add(g, ply)
    return Corpus(n, prefixes, classes, og)


def assignment(P, E, seed):
    """Env -> corpus position: [0, P) in order, then a seeded random draw for [P, E)."""
    rs = np.random.default_rng(seed)
    return np.concatenate([np.arange(P, dtype=np.int64), rs.integers(0, P, E - P, dtype=np.int64)])


def fill(batch, c, src, device_ids):
    """import_state puts the corpus into envs [0, P); clone_gather fills [P, E) by the assignment."""
    batch.import_state(c.records, 0)
    ids = src[c.P:]
    if device_ids:
        import torch
        ids = torch.from_numpy(ids).to("cuda:0")
    batch.clone_gather(ids, c.P)


def hardware():
    import torch
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, p.max_threads_per_multi_processor


# ------------------------------------------------------------------------ the API kernels ---
LIST_ENVS = 30_000
OBS_ENVS = 4_000


@pytest.mark.parametrize("n", SIZES)
def test_list_mask_queries_observation_past_one_pass(n):
    """Legal list (three widths, aligned / unaligned stride and base, odd-first sub-range), legal mask (host,
    device, misaligned device: fast and byte paths), the queries and the observation (+ mask, through the
    producer and DLPack, aligned and misaligned) over several resident passes; every env equals its corpus
    position."""
    import torch
    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.producer import ObservationMaskProducer
    sms, threads_per_sm = hardware()
    assert LIST_ENVS >= 3 * sms * (threads_per_sm // 32)  # >= 3 passes of one warp per env, whatever the occupancy
    assert OBS_ENVS >= 3 * sms * (threads_per_sm // 256)  # >= 3 passes of one 256-thread block per env
    c = corpus(n)
    E = LIST_ENVS
    src = assignment(c.P, E, SEED + n)
    batch = TwixTBatch(n, E, 0, SEED)
    fill(batch, c, src, device_ids=(n % 2 == 0))
    assert np.array_equal(batch.export_state(), c.records[src])
    dev = torch.device("cuda", 0)
    # ---- legal list
    m = batch.max_legal_actions
    assert m == c.legal.shape[1]
    want_cnt = c.counts[src]
    want_list = c.legal[src]
    valid = np.arange(m)[None, :] < want_cnt[:, None]
    for dtype in (torch.int16, torch.int32, torch.int64):
        fill_v = -7
        per_vec = 16 // torch.empty(0, dtype=dtype).element_size()
        aligned = -(-m // per_vec) * per_vec
        want = np.where(valid, want_list, fill_v)
        for stride, off in ((aligned, 0), (aligned + 1, 0), (aligned, 1)):
            flat = torch.full((E * stride + 8,), fill_v, dtype=dtype, device=dev)
            out = flat[off:off + E * stride].view(E, stride)
            cnt = torch.full((E,), -1, dtype=torch.int32, device=dev)
            batch.legal_actions(out_actions=out, out_counts=cnt)
            got = out.cpu().numpy()
            assert np.array_equal(cnt.cpu().numpy(), want_cnt), (n, dtype, stride, off)
            assert np.array_equal(got[:, :m], want), (n, dtype, stride, off)
            assert (got[:, m:] == fill_v).all(), (n, dtype, stride, off)
            edge = flat.cpu().numpy()
            assert (edge[:off] == fill_v).all() and (edge[off + E * stride:] == fill_v).all()
        # a sub-range whose first env is odd (every env's row then lands at a different multiple of the stride)
        first, count = 1001, E - 1001 - 17
        flat = torch.full((count * aligned,), fill_v, dtype=dtype, device=dev)
        cnt = torch.zeros(count, dtype=torch.int32, device=dev)
        batch.legal_actions(first, count, out_actions=flat.view(count, aligned), out_counts=cnt)
        got = flat.view(count, aligned).cpu().numpy()
        assert np.array_equal(cnt.cpu().numpy(), want_cnt[first:first + count]), (n, dtype)
        assert np.array_equal(got[:, :m], want[first:first + count]) and (got[:, m:] == fill_v).all(), (n, dtype)
    la, cnt = batch.legal_actions()  # host int64 output
    assert np.array_equal(cnt, want_cnt) and np.array_equal(np.where(valid, la, -1), want_list)
    # ---- legal mask: host, device aligned and device misaligned (n % 4 == 0: fast path, then byte path)
    want_mask = c.mask[src]
    assert np.array_equal(batch.legal_mask(), want_mask), n
    out = torch.full((E, n * n), 9, dtype=torch.uint8, device=dev)
    batch.legal_mask(out=out)
    assert np.array_equal(out.cpu().numpy(), want_mask), n
    raw = torch.full((E * n * n + 1,), 9, dtype=torch.uint8, device=dev)
    batch.legal_mask(out=raw[1:])
    got = raw.cpu().numpy()
    assert got[0] == 9 and np.array_equal(got[1:].reshape(E, n * n), want_mask), n
    # ---- queries
    assert np.array_equal(batch.current_player(), c.player[src])
    assert np.array_equal(batch.is_terminal(), c.terminal[src])
    assert np.array_equal(batch.returns(), c.returns[src])
    # ---- observation and observation + mask over OBS_ENVS envs
    EO = OBS_ENVS
    osz = 12 * n * (n - 2)
    want_obs = c.obs[src]
    assert np.array_equal(batch.observation(0, EO).reshape(EO, osz), want_obs[:EO]), n  # host output
    f1 = E - EO - 5
    raw = torch.full((EO * osz + 1,), -3.0, dtype=torch.float32, device=dev)  # off the 16-byte grid: scalar path
    batch.observation(f1, EO, out=raw[1:])
    got = raw.cpu().numpy()
    assert got[0] == -3.0 and np.array_equal(got[1:].reshape(EO, osz), want_obs[f1:f1 + EO]), n
    f2 = 7
    o_al = torch.empty((EO, osz), dtype=torch.float32, device=dev)
    m_raw = torch.full((EO * n * n + 3,), 9, dtype=torch.uint8, device=dev)
    batch.observation_and_mask(f2, EO, out_obs=o_al, out_mask=m_raw[3:])
    assert np.array_equal(o_al.cpu().numpy(), want_obs[f2:f2 + EO]), n
    got = m_raw.cpu().numpy()
    assert (got[:3] == 9).all() and np.array_equal(got[3:].reshape(EO, n * n), want_mask[f2:f2 + EO]), n
    raw = torch.full((EO * osz + 1,), -3.0, dtype=torch.float32, device=dev)
    m_al = torch.empty((EO, n * n), dtype=torch.uint8, device=dev)
    batch.observation_and_mask(f1, EO, out_obs=raw[1:], out_mask=m_al)
    assert np.array_equal(raw[1:].cpu().numpy().reshape(EO, osz), want_obs[f1:f1 + EO]), n
    assert np.array_equal(m_al.cpu().numpy(), want_mask[f1:f1 + EO]), n
    prod = ObservationMaskProducer(batch, max_count=EO)
    f3 = E - EO
    obs_t, mask_t = prod.produce(f3, EO)
    assert np.array_equal(obs_t.cpu().numpy().reshape(EO, osz), want_obs[f3:]), n
    assert np.array_equal(mask_t.cpu().numpy(), want_mask[f3:]), n
    f4, k4 = 12_345, EO - 3
    cap_obs, cap_mask = prod.produce_dlpack(f4, k4)
    o2, m2 = torch.from_dlpack(cap_obs), torch.from_dlpack(cap_mask)
    assert np.array_equal(o2.cpu().numpy().reshape(k4, osz), want_obs[f4:f4 + k4]), n
    assert np.array_equal(m2.cpu().numpy(), want_mask[f4:f4 + k4]), n
    batch.close()


CLONE_ENVS = 150_000
CLONE_GRID_QUADS = 148 * 64 * 256  # twixt_kernels_api.cu: grid_for caps reset / clone at 148 x 64 blocks of 256


def test_clone_gather_clone_reset_past_one_grid_pass(oracle_mod):
    """reset / clone / clone_gather at n = 24 over ranges of more 16-byte quads than one grid pass covers:
    exports equal the gathered corpus records, and a reset sub-range leaves its neighbours alone."""
    from twixt_for_open_spiel_b200 import TwixTBatch
    n, E = 24, CLONE_ENVS
    c = corpus(n)
    quads = c.records.shape[1] // 4
    half = E // 2
    assert (E - c.P) * quads > 2 * CLONE_GRID_QUADS and half * quads > CLONE_GRID_QUADS
    src = assignment(c.P, E, SEED + 424)
    batch = TwixTBatch(n, E, 0, SEED)
    fill(batch, c, src, device_ids=True)
    recs = batch.export_state()
    assert np.array_equal(recs, c.records[src])
    batch.clone(half, 0, half)  # the second half over the first
    after = batch.export_state()
    assert np.array_equal(after[:half], recs[half:]) and np.array_equal(after[half:], recs[half:])
    batch.clone(0, half, half)  # and back: the first half over the second
    after = batch.export_state()
    assert np.array_equal(after, np.concatenate([recs[half:], recs[half:]]))
    init = oracle_mod.OracleGame(n).new_initial_state().export_record()
    first, count = 3, E - 3 - 5
    assert count * quads > CLONE_GRID_QUADS
    batch.reset(first, count)
    done = batch.export_state()
    assert (done[first:first + count] == init[None, :]).all()
    assert np.array_equal(done[:first], after[:first]) and np.array_equal(done[first + count:], after[first + count:])
    batch.close()


VALIDATE_ENVS = 60_000
VALIDATE_WARPS = 148 * 16 * 8  # twixt_kernels_api.cu: launch_validate's grid cap x 8 warps per block


@pytest.mark.parametrize("n", [5, 13, 24])
def test_import_validation_past_one_pass(n):
    """import_state validates E corpus records over several grid-stride passes: all are accepted; two corrupt
    records past the first pass are reported by the LOWER index and change nothing; a bad last record is
    found."""
    import torch
    from twixt_for_open_spiel_b200 import TwixTBatch
    assert VALIDATE_ENVS >= 3 * VALIDATE_WARPS
    c = corpus(n)
    E = VALIDATE_ENVS
    good = c.records[assignment(c.P, E, SEED + 5 * n)]
    batch = TwixTBatch(n, E, 0, SEED)
    batch.import_state(good)
    assert np.array_equal(batch.export_state(), good)
    lo, hi = VALIDATE_WARPS + 5_000, 2 * VALIDATE_WARPS + 100  # second and third pass, hi by a lower warp
    bad = good.copy()
    bad[hi, 4 + 1] |= np.uint32(1 << n)  # a red bit on row n ("rows")
    bad[lo, 3] += np.uint32(1)           # the empty-cell count ("counts")
    batch.reset()
    before = batch.export_state()
    for device_side in (False, True):
        srcr = torch.from_numpy(bad.view(np.int32)).to("cuda:0") if device_side else bad
        with pytest.raises(ValueError) as err:
            batch.import_state(srcr)
        assert str(err.value).startswith("invalid state record at index %d:" % lo), str(err.value)
        assert "counts" in str(err.value)
        assert np.array_equal(batch.export_state(), before)
    last = good.copy()
    last[E - 1, 3] += np.uint32(1)
    with pytest.raises(ValueError, match=r"^invalid state record at index %d:" % (E - 1)):
        batch.import_state(last)
    assert np.array_equal(batch.export_state(), before)
    batch.close()


# -------------------------------------------------------------------------- playout tickets ---
_LAUNCH = re.compile(r"\[twixt_b200\] playout n=(\d+): (\d+) blocks x (\d+) threads")
TICKET_FREE_ENVS = 8_192  # <= 64 blocks of >= 128 threads: fewer than one resident wave, no ticket is taken


def launches(capfd):
    """(n, blocks, threads) of every playout launch since the last call (TWIXT_B200_DEBUG=1 lines)."""
    err = capfd.readouterr().err
    return [tuple(int(v) for v in m.groups()) for m in _LAUNCH.finditer(err)]


def _expected_stats(start, final, lens):
    """stats() totals implied by the starting and final records and the lengths of one playout call."""
    res0, res1 = start[:, 1] & 3, final[:, 1] & 3
    games = (res0 == KOPEN) & (res1 != KOPEN)
    return {"games": int(games.sum()), "plies": int(lens.astype(np.int64).sum()),
            "red_wins": int((games & (res1 == KRED)).sum()), "blue_wins": int((games & (res1 == KBLUE)).sum()),
            "draws": int((games & (res1 == KDRAW)).sum()),
            "swaps": int((((start[:, 1] >> 2) & 1) != ((final[:, 1] >> 2) & 1)).sum()),
            "max_length": int(final[games, 0].max()) if games.any() else 0}


def _ticket_free(n, start, streams, budget, trace_rows, capfd):
    """The same starting records and streams played in launches of <= TICKET_FREE_ENVS envs (each launch
    checked to take no ticket): (returns, lengths, final records, trace)."""
    from twixt_for_open_spiel_b200 import TwixTBatch
    E = start.shape[0]
    ref = TwixTBatch(n, TICKET_FREE_ENVS, 0, SEED)
    ref.set_validation(False)  # corpus records, validated elsewhere
    rets = np.zeros((E, 2), dtype=np.float32)
    lens = np.zeros(E, dtype=np.int32)
    recs = np.zeros_like(start)
    trace = np.zeros((trace_rows, E), dtype=np.uint16) if trace_rows else None
    for a in range(0, E, TICKET_FREE_ENVS):
        k = min(TICKET_FREE_ENVS, E - a)
        ref.import_state(start[a:a + k])
        out_act = np.zeros((trace_rows, k), dtype=np.uint16) if trace_rows else None
        r, ln, tr = ref.playout(0, k, max_plies=budget, stream_ids=streams[a:a + k], out_actions=out_act)
        (ln_n, blocks, threads), = launches(capfd)
        assert ln_n == n and blocks * threads >= k  # every env pre-assigned: no tickets
        rets[a:a + k], lens[a:a + k], recs[a:a + k] = r, ln, ref.export_state(0, k)
        if trace_rows:
            trace[:, a:a + k] = tr
    ref.close()
    return rets, lens, recs, trace


def _oracle_check(c, src, streams, budget, rets, lens, recs, trace, envs):
    for e in envs:
        st = c.state(int(src[e]))
        acts = st.playout_philox(SEED, int(streams[e]), budget)
        assert lens[e] == len(acts), e
        assert np.array_equal(recs[e], st.export_record()), e
        assert rets[e].tolist() == st.returns(), e
        if trace is not None:
            t = min(len(acts), trace.shape[0])
            assert trace[:t, e].tolist() == acts[:t] and (trace[t:, e] == 0xFFFF).all(), e


TRACED_SIZES = (5, 13, 24)


@pytest.mark.parametrize("n", SIZES)
def test_playout_tickets_with_the_product_grid(n, monkeypatch, capfd):
    """E = 2 x (the product grid's lanes) + 123 envs from the corpus, so about half of them are taken by
    ticket, with stream_base, host uint64 ids, device int64 ids and a ply budget (and a truncated trace at
    three sizes): every env bit-identical to ticket-free launches of the same starts, the last 1 024 tickets
    and ~1 000 random envs replayed on the oracle, stats() equal to what the outputs imply."""
    import torch
    from twixt_for_open_spiel_b200 import TwixTBatch
    monkeypatch.setenv("TWIXT_B200_DEBUG", "1")
    capfd.readouterr()
    sms, threads_per_sm = hardware()
    assert TICKET_FREE_ENVS <= 64 * 128 and 64 < sms
    probe = TwixTBatch(n, sms * threads_per_sm, 0, SEED)  # more envs than lanes can be resident
    probe.playout(max_plies=0, want_returns=False, want_lengths=False)
    probe.close()
    (pn, blocks, threads), = launches(capfd)
    assert pn == n
    E = 2 * blocks * threads + 123
    c = corpus(n)
    src = assignment(c.P, E, SEED + 31 * n)
    start = c.records[src]
    batch = TwixTBatch(n, E, 0, SEED)
    rs = np.random.default_rng(n)
    sample = sorted(set(range(E - 1024, E)) | set(rs.integers(0, E - 1024, 1000).tolist()))
    budget_small = max(3, (n * n) // 4)
    calls = [("stream_base", None), ("host_ids", None), ("device_ids", budget_small)]
    if n in TRACED_SIZES:
        calls.append(("traced", None))
    for name, budget in calls:
        fill(batch, c, src, device_ids=(name == "device_ids"))
        batch.stats_reset()
        launches(capfd)  # (nothing launched the playout kernel since)
        base = 0
        if name in ("stream_base", "traced"):
            base = 1_000_003 * n + (7 if name == "traced" else 0)
            batch.set_stream_base(base)
            streams = base + np.arange(E, dtype=np.uint64)
            ids = None
        else:
            streams = rs.integers(0, 1 << 62, E, dtype=np.int64).astype(np.uint64)
            ids = streams if name == "host_ids" else torch.from_numpy(streams.view(np.int64)).to("cuda:0")
        trace_rows = (n * n) // 3 if name == "traced" else 0
        out_act = np.zeros((trace_rows, E), dtype=np.uint16) if trace_rows else None
        mp = budget if budget is not None else n * n
        rets, lens, trace = batch.playout(max_plies=mp, stream_ids=ids, out_actions=out_act)
        (ln, lb, lt), = launches(capfd)
        assert (ln, lb, lt) == (n, blocks, threads) and lb < -(-E // lt), name  # tickets were taken
        batch.set_stream_base(0)
        recs = batch.export_state()
        st = batch.stats()
        # terminal starts come back unchanged, with length 0
        term = c.terminal[src].astype(bool)
        assert term.sum() > 0 and (lens[term] == 0).all() and np.array_equal(recs[term], start[term]), name
        want = _expected_stats(start, recs, lens)
        assert {k: st[k] for k in want} == want, (name, st, want)
        if budget is None:
            assert ((recs[:, 1] & 3) != KOPEN).all(), name
        else:
            assert (lens <= budget).all() and (lens == budget).any(), name
        tr, tl, trec, ttrace = _ticket_free(n, start, streams, mp, trace_rows, capfd)
        assert np.array_equal(lens, tl), name
        assert np.array_equal(rets, tr), name
        assert np.array_equal(recs, trec), name
        if trace_rows:
            assert np.array_equal(trace, ttrace), name
            full = lens <= trace_rows
            assert full.any() and (~full).any()  # complete and truncated trace rows
        _oracle_check(c, src, streams, mp, rets, lens, recs, trace, sample)
    batch.close()


# ---------------------------------------------------------------- deep ticket chains (variant) ---
CHAIN_ENVS = 3_400  # >= 10 envs per lane at the widest block (320 threads)


def chain_main():
    """Run in a subprocess against the TW_PLAYOUT_MAX_BLOCKS=1 build: one block plays every env, so each lane
    plays ten or more games in a row; every env of every call is compared with the oracle, and a device MCTS
    search (whose rollout launches take tickets with the search's own stream ids) with its specification."""
    import mcts_spec as spec
    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    for n in SIZES:
        c = corpus(n)
        E = CHAIN_ENVS
        src = assignment(c.P, E, SEED + 97 * n)
        b = TwixTBatch(n, E, 0, SEED)
        rs = np.random.default_rng(1000 + n)
        for budget in (None, max(3, (n * n) // 4)):
            fill(b, c, src, device_ids=(budget is None))
            streams = rs.integers(0, 1 << 62, E, dtype=np.int64).astype(np.uint64)
            mp = budget if budget is not None else n * n
            rets, lens, trace = b.playout(max_plies=mp, stream_ids=streams, trace=budget is None)
            recs = b.export_state()
            _oracle_check(c, src, streams, mp, rets, lens, recs, trace, range(E))
        b.close()
        print("chain n=%d ok" % n, flush=True)
    n, trees, sims, R = 8, 64, 100, 8
    from oracle import pyoracle
    g = pyoracle.OracleGame(n)
    roots = spec.root_positions(g, n, 11, trees)
    b = TwixTBatch(n, trees, 0, SEED)
    b.import_state(np.stack([r.export_record() for r in roots]), 0)
    b.set_stream_base(100)
    m = BatchedMCTS(b, trees, sims, R, 1.5)
    m.begin(0, trees)
    m.run(sims)
    visits, sums, best = m.root_stats()
    for t, r in enumerate(roots):
        v, w, bst = spec.Search(r, SEED, 100 + t, R, 1.5).run(sims).root_stats(n)
        assert np.array_equal(visits[t], v) and sums[t].tobytes() == w.tobytes() and best[t] == bst, t
    print("chain ok", flush=True)


def test_playout_deep_ticket_chains_with_one_block():
    """The playout kernel built with TW_PLAYOUT_MAX_BLOCKS=1: all 20 sizes, corpus starts, explicit ids, a
    traced and a budgeted run, every env against the oracle; one device MCTS search against mcts_spec.py.
    Every launch ran on exactly one block."""
    from twixt_for_open_spiel_b200 import build
    variant = build.build(out=os.path.join(HERE, "_build", "libtwixt_b200_tickets.so"),
                          extra_flags=["-DTW_PLAYOUT_MAX_BLOCKS=1"])
    code = "import sys; sys.path[:0] = [%r, %r]; import test_gpu_multipass as t; t.chain_main()" % (HERE, ROOT)
    env = dict(os.environ, TWIXT_B200_LIB=variant, TWIXT_B200_DEBUG="1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT)
    assert res.returncode == 0 and "chain ok" in res.stdout, (res.stdout[-500:], res.stderr[-3000:])
    grid = [tuple(int(v) for v in m.groups()) for m in _LAUNCH.finditer(res.stderr)]
    assert len(grid) >= 2 * len(SIZES) + 100  # two calls per size + one rollout launch per MCTS simulation step
    assert all(blocks == 1 for _, blocks, _ in grid), sorted(set(grid))[:5]
    assert all(CHAIN_ENVS >= 10 * threads for _, _, threads in grid)
