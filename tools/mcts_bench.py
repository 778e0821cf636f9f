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
                 endgame: bool = False) -> dict:
    import torch
    from torch.profiler import ProfilerActivity, profile

    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    b = endgame_roots(n, trees, 0x736F6C76) if endgame else make_roots(n, trees, 0x6D637473)
    m = BatchedMCTS(b, trees, sims, R, solve=solve)
    # warm-up: every kernel of a simulation, at this size
    m.begin(0, trees)
    m.run(min(sims, 20))
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
        "ms_per_simulation_step": round(ms / sims, 4),
        "kernel_ms_per_simulation_step": {k: round(v / 1e3 / profile_sims, 4) for k, v in split.items()},
        "roots_with_a_best_move": int((best >= 0).sum()),
    }
    if solve:
        proven, _, _, simulations = solved
        out.update({"solve": True, "roots": "endgame" if endgame else "opening",
                    "fraction_proven": round(float(proven.mean()), 4),
                    "mean_root_visits": round(float(simulations.mean()), 2)})
    return out


def bench_puct(n: int, trees: int, sims: int, profile_sims: int) -> dict:
    import torch
    from torch.profiler import ProfilerActivity, profile

    from twixt_for_open_spiel_b200.mcts import BatchedMCTS
    b = make_roots(n, 2 * trees, 0x70756374)  # envs [trees, 2*trees) take the leaves
    m = BatchedMCTS(b, trees, sims, selection="puct")
    gen = torch.Generator(device="cuda").manual_seed(1)
    priors = torch.rand((trees, n * n), generator=gen, device="cuda", dtype=torch.float32)
    values = torch.zeros((trees, 2), device="cuda", dtype=torch.float32)
    status = torch.zeros(trees, dtype=torch.int32, device="cuda")

    def search(k):
        for _ in range(k):
            m.select(trees, status)
            m.backup(values, priors)

    m.begin(0, trees)
    search(min(sims, 20))
    b.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m.begin(0, trees)
    start.record()
    search(sims)
    stop.record()
    stop.synchronize()
    ms = start.elapsed_time(stop)
    m.begin(0, trees)
    b.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        search(profile_sims)
        b.synchronize()
    split = {"select": 0.0, "backup": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if "mcts_select_kernel" in ev.key:
            split["select"] += t
        elif "mcts_backup_kernel" in ev.key:
            split["backup"] += t
    best = m.best()
    m.close()
    b.close()
    return {
        "board_size": n, "trees": trees, "simulations": sims,
        "search_ms": round(ms, 3),
        "simulations_per_s": round(trees * sims / (ms / 1e3), 1),
        "ms_per_simulation_step": round(ms / sims, 4),
        "kernel_ms_per_simulation_step": {k: round(v / 1e3 / profile_sims, 4) for k, v in split.items()},
        "roots_with_a_best_move": int((best >= 0).sum()),
    }


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
    else:
        configs = [(12, 8192, 400, 4, 50), (24, 1024, 200, 4, 50)]
        puct = [(12, 8192, 400, 50), (24, 1024, 200, 50)]
        ev = (12, 8192, 4, 50)
        solve = [(12, 8192, 400, 4, 50, True, False), (8, 8192, 400, 4, 50, True, True)]
    out = dict(info)
    out["configs"] = [bench_config(*c) for c in configs]
    out["evaluate_slots"] = bench_evaluator(*ev)
    out["puct"] = [bench_puct(*c) for c in puct]
    if not args.no_solve:
        out["solve"] = [bench_config(*c) for c in solve]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
