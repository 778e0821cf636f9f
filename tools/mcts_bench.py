"""Throughput of the batched device MCTS (twixt_for_open_spiel_b200/mcts.py); prints ONE JSON line.

    python tools/mcts_bench.py [--quick]

Two configurations, each from roots a few random plies into a game (seeded):
  n = 12: 8192 trees x 400 simulations x R = 4 rollouts
  n = 24: 1024 trees x 200 simulations x R = 4
For each: simulations/s (tree-simulations per second over all trees) and rollout plies/s of a whole warmed-up
search timed with CUDA events, and the ms per simulation step spent in select / playout / backup kernels,
from torch.profiler over a separate run of the same search.  BatchedRolloutEvaluator.evaluate_slots leaves/s
at n = 12 (8192 leaves x R = 4) is on the same line as the reference point.  The device name and power limit
are read in the same process.

`puct`: the stepwise PUCT search (selection="puct", select -> backup(values, priors)) with a fixed
device-resident prior tensor (seeded uniform random, so score ties are as rare as with a network) and zero
values, so that the search itself is measured and no network:
  n = 12: 8192 trees x 400 simulations;  n = 24: 1024 trees x 200
with simulations/s and the select / backup kernel ms per step, next to the UCT configurations above.

`solve`: the MCTS-Solver (solve=True, UCT with rollouts):
  n = 12: the first UCT configuration above with solve=True: the solver's overhead where little gets proven;
  n = 8 endgames: 8192 roots 2..6 plies before the end of seeded games x 400 simulations x R = 4, where most
  trees finish early; simulations/s counts every tree's simulations (finished ones too), next to the fraction of
  roots proven, the mean N(root) and the backup kernel ms per step.

`parallel`: several leaves per step with virtual loss (leaves_per_step = K, virtual_loss = 1):
  one tree at n = 12 x 1000 simulations x R = 4 (an MCTSBot.step-sized search) at K = 1, 8 and 32 (992
  simulations there, whole steps): wall time per search (begin + run, ending in a device synchronise), mean of 5
  after a warm-up;
  64 trees x 400 simulations at n = 12, UCT x R = 4 (run) and the stepwise PUCT search above, at K = 1 and 8:
  simulations/s and the select / playout / backup kernel ms per step (a step is K simulations of every tree).

`reuse`: tree reuse across moves (BatchedMCTS.advance):
  the advance kernel alone at n = 12 for 8192 stepwise PUCT trees after a 400-simulation search (capacity 800,
  keep 401), along each tree's best move: device ms (torch.profiler, mean of 3 searches) and an estimate of the
  bytes it moves (each kept node's record, counts and L edges read and written once, L the root's legal count, the
  kept nodes N(new root)), as GB/s and a fraction of the 7.7 TB/s HBM3e peak of one HGX B200 GPU (data sheet);
  a multi-move loop of the stepwise PUCT search above (1024 trees at n = 12, 100 new simulations per move, 12
  moves along the best move) with begin every move and with advance(best, 101) on a capacity of 200: moves/s and
  the mean N(root) at the start of each move's search (sum of the root's N(a) + 1 for an expanded root).
  Both use seeded uniform random priors raised to the 8th power, so that a few moves carry most of a node's prior
  as with a trained policy (flat priors spread the visits over all moves and leave little to keep), and zero values.

`gumbel`: the stepwise Gumbel AlphaZero search (selection="gumbel", max_considered = 16, select -> backup(values,
logits)) with fixed device-resident logits (seeded standard normal), zero values and fresh root Gumbel noise per
search, and next to each entry the stepwise PUCT search above at the same size, in the same process:
  n = 12: 8192 trees x 16, 64 and 400 simulations;  n = 24: 1024 trees x 200
with simulations/s and the select / backup kernel ms per step.  `--gumbel-only` runs just these entries.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def device_info() -> dict:
    import torch
    info = {"device": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")[:2]]
        info["device"] = name
        info["power_limit_w"] = float(limit)
    except Exception:
        pass
    return info


def make_roots(n: int, trees: int, seed: int):
    from twixt_for_open_spiel_b200 import TwixTBatch
    b = TwixTBatch(n, trees, 0, seed)
    b.use_torch_stream()
    b.playout(0, trees, max_plies=6, want_returns=False, want_lengths=False)
    return b


def endgame_roots(n: int, trees: int, seed: int):
    from twixt_for_open_spiel_b200 import TwixTBatch
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    try:
        from mcts_solver import endgame_roots as make
    finally:
        sys.path.pop(0)
    b = TwixTBatch(n, trees, 0, seed)
    make(b, 0, trees)
    b.use_torch_stream()
    return b


def bench_config(n: int, trees: int, sims: int, R: int, profile_sims: int, solve: bool = False,
                 endgame: bool = False, leaves_per_step: int = 1) -> dict:
    import torch
    from torch.profiler import ProfilerActivity, profile

    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    K = leaves_per_step
    b = endgame_roots(n, trees, 0x736F6C76) if endgame else make_roots(n, trees, 0x6D637473)
    m = BatchedMCTS(b, trees, sims, R, solve=solve, leaves_per_step=K)
    # warm-up: every kernel of a simulation, at this size
    m.begin(0, trees)
    m.run(max(K, min(sims, 20) // K * K))
    b.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0 = b.stats()["plies"]
    m.begin(0, trees)
    start.record()
    m.run(sims)
    stop.record()
    stop.synchronize()
    ms = start.elapsed_time(stop)
    plies = b.stats()["plies"] - p0
    solved = m.solver_stats() if solve else None
    # the split, from the kernels' device time in a separate profiled run
    m.begin(0, trees)
    b.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.run(profile_sims)
        b.synchronize()
    split = {"select": 0.0, "playout": 0.0, "backup": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        name = ev.key
        if "mcts_select_kernel" in name:
            split["select"] += t
        elif "mcts_backup_kernel" in name:
            split["backup"] += t
        elif "playout" in name:
            split["playout"] += t
    best = m.best()
    m.close()
    b.close()
    out = {
        "board_size": n, "trees": trees, "simulations": sims, "n_rollouts": R,
        "search_ms": round(ms, 3),
        "simulations_per_s": round(trees * sims / (ms / 1e3), 1),
        "rollout_plies_per_s": round(plies / (ms / 1e3), 1),
        "ms_per_simulation_step": round(ms / (sims // K), 4),
        "kernel_ms_per_simulation_step": {k: round(v / 1e3 / (profile_sims // K), 4) for k, v in split.items()},
        "roots_with_a_best_move": int((best >= 0).sum()),
    }
    if K > 1:
        out["leaves_per_step"] = K
    if solve:
        proven, _, _, simulations = solved
        out.update({"solve": True, "roots": "endgame" if endgame else "opening",
                    "fraction_proven": round(float(proven.mean()), 4),
                    "mean_root_visits": round(float(simulations.mean()), 2)})
    return out


def bench_puct(n: int, trees: int, sims: int, profile_sims: int, leaves_per_step: int = 1,
               selection: str = "puct") -> dict:
    import torch
    from torch.profiler import ProfilerActivity, profile

    from twixt_for_open_spiel_b200.mcts import BatchedMCTS, gumbel_noise
    K = leaves_per_step
    rows = trees * K
    gumbel = selection == "gumbel"
    b = make_roots(n, trees + rows, 0x70756374)  # envs [trees, trees + trees*K) take the leaves
    m = BatchedMCTS(b, trees, sims, selection=selection, leaves_per_step=K)
    gen = torch.Generator(device="cuda").manual_seed(1)
    if gumbel:  # logits
        priors = torch.randn((rows, n * n), generator=gen, device="cuda", dtype=torch.float32)
    else:
        priors = torch.rand((rows, n * n), generator=gen, device="cuda", dtype=torch.float32)
    values = torch.zeros((rows, 2), device="cuda", dtype=torch.float32)
    status = torch.zeros(rows, dtype=torch.int32, device="cuda")

    def begin():
        m.begin(0, trees)
        if gumbel:
            m.set_root_gumbel(gumbel_noise(trees, n * n, generator=gen, device="cuda"))

    def search(k):  # k simulations of every tree: k / K steps
        for _ in range(k // K):
            m.select(trees, status)
            m.backup(values, priors)

    begin()
    search(max(K, min(sims, 20) // K * K))
    b.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    begin()
    start.record()
    search(sims)
    stop.record()
    stop.synchronize()
    ms = start.elapsed_time(stop)
    begin()
    b.synchronize()
    profile_sims = min(profile_sims, sims)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        search(profile_sims)
        b.synchronize()
    split = {"select": 0.0, "backup": 0.0}
    names = ("mcts_gumbel_select_kernel", "mcts_gumbel_backup_kernel") if gumbel else ("mcts_select_kernel",
                                                                                      "mcts_backup_kernel")
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if names[0] in ev.key:
            split["select"] += t
        elif names[1] in ev.key:
            split["backup"] += t
    best = m.best()
    m.close()
    b.close()
    out = {
        "selection": selection, "board_size": n, "trees": trees, "simulations": sims,
        "search_ms": round(ms, 3),
        "simulations_per_s": round(trees * sims / (ms / 1e3), 1),
        "ms_per_simulation_step": round(ms / (sims // K), 4),
        "kernel_ms_per_simulation_step": {k: round(v / 1e3 / (profile_sims // K), 4) for k, v in split.items()},
        "roots_with_a_best_move": int((best >= 0).sum()),
    }
    if K > 1:
        out["leaves_per_step"] = K
    return out


def bench_single_tree(n: int, sims: int, R: int, K: int, reps: int) -> dict:
    """One tree, the search of one MCTSBot.step: wall time of begin + run(sims), ending in a synchronise.  sims is
    rounded down to a multiple of K (run takes whole steps): 992 at K = 32 for 1000."""
    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    sims -= sims % K
    b = make_roots(n, 1, 0x626F7473)
    m = BatchedMCTS(b, 1, sims, R, leaves_per_step=K)
    m.begin(0, 1)
    m.run(sims)
    b.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        m.begin(0, 1)
        m.run(sims)
        b.synchronize()
        times.append(time.perf_counter() - t0)
    m.close()
    b.close()
    return {"board_size": n, "trees": 1, "simulations": sims, "n_rollouts": R, "leaves_per_step": K,
            "steps": sims // K, "ms_per_search": round(1e3 * sum(times) / reps, 3),
            "ms_per_search_min": round(1e3 * min(times), 3)}


def _puct_steps(m, trees, sims, values, priors, status):
    for _ in range(sims):
        m.select(trees, status)
        m.backup(values, priors)


def bench_advance(n: int, trees: int, sims: int, reps: int) -> dict:
    import torch
    from torch.profiler import ProfilerActivity, profile

    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    b = make_roots(n, 2 * trees, 0x72757365)
    m = BatchedMCTS(b, trees, 2 * sims, selection="puct")
    gen = torch.Generator(device="cuda").manual_seed(2)
    priors = torch.rand((trees, n * n), generator=gen, device="cuda", dtype=torch.float32) ** 8  # peaked
    values = torch.zeros((trees, 2), device="cuda", dtype=torch.float32)
    status = torch.zeros(trees, dtype=torch.int32, device="cuda")
    visits = torch.zeros((trees, n * n), dtype=torch.int32, device="cuda")
    best = torch.zeros(trees, dtype=torch.int32, device="cuda")
    rw = b.record_words
    kernel_us, kept_total, edge_bytes = [], 0, 0
    for rep in range(reps + 1):  # the first is a warm-up
        m.begin(0, trees)
        _puct_steps(m, trees, sims, values, priors, status)
        m.root_stats(out_visits=visits, out_best=best)
        b.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m.advance(best, sims + 1, out_status=status)
            b.synchronize()
        if rep == 0:
            continue
        kernel_us.append(sum(getattr(ev, "device_time_total", None) or ev.cuda_time_total
                             for ev in prof.key_averages() if "mcts_advance_kernel" in ev.key))
        kept = visits.gather(1, best.clamp_min(0).long()[:, None])[:, 0].long()  # N(a) of the move = kept nodes
        _, cnt = b.legal_actions(0, trees)  # the old roots' legal counts
        L = torch.as_tensor(cnt, device="cuda").long()
        kept_total = int(kept.sum())
        # per kept node: record + legal count + N(s) + L edges (action 2, N 4, W 8, child 4, prior 4, key 4,
        # outcome 1) read and written, and the slot map written and read
        edge_bytes = int((kept * (2 * (rw * 4 + 8 + 27 * L) + 8)).sum())
    ms = sum(kernel_us) / len(kernel_us) / 1e3
    m.close()
    b.close()
    gbs = edge_bytes / (ms / 1e3) / 1e9
    return {"board_size": n, "trees": trees, "simulations": sims, "capacity": 2 * sims, "keep_nodes": sims + 1,
            "advance_kernel_ms": round(ms, 4), "kept_nodes": kept_total, "estimated_bytes_moved": edge_bytes,
            "estimated_gb_per_s": round(gbs, 1), "fraction_of_hbm_peak": round(gbs / 7700.0, 4)}


def bench_moves(n: int, trees: int, sims: int, moves: int, reuse: bool) -> dict:
    import torch

    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    b = make_roots(n, 2 * trees, 0x6D6F7665)
    start_records = b.export_state(0, trees)
    m = BatchedMCTS(b, trees, 2 * sims, selection="puct")
    gen = torch.Generator(device="cuda").manual_seed(3)
    priors = torch.rand((trees, n * n), generator=gen, device="cuda", dtype=torch.float32) ** 8  # peaked
    values = torch.zeros((trees, 2), device="cuda", dtype=torch.float32)
    status = torch.zeros(trees, dtype=torch.int32, device="cuda")
    visits = torch.zeros((trees, n * n), dtype=torch.int32, device="cuda")
    best = torch.zeros(trees, dtype=torch.int32, device="cuda")
    root_n = torch.zeros(moves, dtype=torch.float64, device="cuda")

    def play(record_n):
        m.begin(0, trees)
        for mv in range(moves):
            if mv > 0 and not reuse:
                m.begin(0, trees)
            if record_n:
                m.root_stats(out_visits=visits)
                total = visits.sum(1)
                root_n[mv] = (total + (total > 0).int()).double().mean()
            _puct_steps(m, trees, sims, values, priors, status)
            m.root_stats(out_best=best)
            b.apply(best, 0)
            if reuse:
                m.advance(best, sims + 1, out_status=status)

    play(False)  # warm-up
    b.import_state(start_records, 0)
    b.synchronize()
    t0 = time.perf_counter()
    play(False)
    b.synchronize()
    dt = time.perf_counter() - t0
    b.import_state(start_records, 0)
    play(True)
    b.synchronize()
    per_move = root_n.cpu().tolist()
    m.close()
    b.close()
    return {"board_size": n, "trees": trees, "new_simulations_per_move": sims, "moves": moves, "reuse_tree": reuse,
            "moves_per_s": round(moves / dt, 2), "simulations_per_s": round(trees * sims * moves / dt, 1),
            "mean_root_visits_at_search_start": round(sum(per_move) / moves, 2),
            "mean_root_visits_by_move": [round(x, 1) for x in per_move]}


def bench_evaluator(n: int, leaves: int, R: int, reps: int) -> dict:
    from twixt_for_open_spiel_b200.rollout import BatchedRolloutEvaluator
    ev = BatchedRolloutEvaluator(n, n_rollouts=R, max_leaves=leaves, seed=1)
    ev.batch.reset()
    ev.batch.playout(0, leaves, max_plies=6, want_returns=False, want_lengths=False)
    ev.evaluate_slots(leaves)
    t0 = time.perf_counter()
    for _ in range(reps):
        ev.evaluate_slots(leaves)  # ends in a device-to-host copy of the means: synchronous
    dt = time.perf_counter() - t0
    ev.close()
    return {"board_size": n, "leaves": leaves, "n_rollouts": R, "leaves_per_s": round(leaves * reps / dt, 1)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="small sizes (a functional check, not a measurement)")
    ap.add_argument("--no-solve", action="store_true", help="skip the solver entries")
    ap.add_argument("--no-parallel", action="store_true", help="skip the leaves_per_step entries")
    ap.add_argument("--no-reuse", action="store_true", help="skip the tree reuse entries")
    ap.add_argument("--gumbel-only", action="store_true", help="only the gumbel entries and their puct pairs")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mcts_bench needs a CUDA device")
    info = device_info()
    if args.quick:
        configs = [(12, 256, 40, 4, 10), (24, 64, 20, 4, 5)]
        puct = [(12, 256, 40, 10), (24, 64, 20, 5)]
        ev = (12, 256, 4, 5)
        solve = [(12, 256, 40, 4, 10, True, False), (8, 256, 40, 4, 10, True, True)]
        single = [(12, 96, 4, K, 2) for K in (1, 8, 32)]
        many = [(12, 16, 48, 4, 16, K) for K in (1, 8)]
        adv = (12, 256, 40, 2)
        moves = (12, 64, 20, 4)
        gumbel = [(12, 256, 16, 16), (12, 256, 64, 20), (24, 64, 20, 10)]
    else:
        configs = [(12, 8192, 400, 4, 50), (24, 1024, 200, 4, 50)]
        puct = [(12, 8192, 400, 50), (24, 1024, 200, 50)]
        ev = (12, 8192, 4, 50)
        solve = [(12, 8192, 400, 4, 50, True, False), (8, 8192, 400, 4, 50, True, True)]
        single = [(12, 1000, 4, K, 5) for K in (1, 8, 32)]
        many = [(12, 64, 400, 4, 80, K) for K in (1, 8)]
        adv = (12, 8192, 400, 3)
        moves = (12, 1024, 100, 12)
        gumbel = [(12, 8192, 16, 16), (12, 8192, 64, 50), (12, 8192, 400, 50), (24, 1024, 200, 50)]
    out = dict(info)
    if args.gumbel_only:
        out["gumbel"] = [[bench_puct(*c, selection=k) for k in ("gumbel", "puct")] for c in gumbel]
        print(json.dumps(out))
        return
    out["configs"] = [bench_config(*c) for c in configs]
    out["evaluate_slots"] = bench_evaluator(*ev)
    out["puct"] = [bench_puct(*c) for c in puct]
    if not args.no_solve:
        out["solve"] = [bench_config(*c) for c in solve]
    if not args.no_parallel:
        out["parallel"] = {
            "single_tree": [bench_single_tree(*c) for c in single],
            "uct": [bench_config(n, t, s, R, p, leaves_per_step=K) for n, t, s, R, p, K in many],
            "puct": [bench_puct(n, t, s, p, leaves_per_step=K) for n, t, s, _, p, K in many],
        }
    if not args.no_reuse:
        out["reuse"] = {"advance": bench_advance(*adv),
                        "moves": [bench_moves(*moves, reuse=r) for r in (False, True)]}
    out["gumbel"] = [[bench_puct(*c, selection=k) for k in ("gumbel", "puct")] for c in gumbel]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
