#!/usr/bin/env python3
"""A/B timing of playout-kernel VARIANT builds on the GPU box (development tool).

    python tools/ab_playout.py build  name=-DFLAG=1,-DOTHER=0 ...   # here (CPU): builds tests/_build/variants/<name>.so
    python tools/ab_playout.py run [n[,n..]] [envs] [reps] [rounds]  # on the GPU box: times every variant found

Each variant runs in its own process (the library is chosen once per process through TWIXT_B200_LIB), is first
checked against the oracle on 96 complete games, then timed with CUDA events on the launching stream: `reps`
launches of reset + playout of `envs` fresh games, each with its own seed; prints min / median ms per launch.
A list of board sizes is timed size by size in each process; the variants alternate for `rounds` rounds
(default 2)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VDIR = os.path.join(ROOT, "tests", "_build", "variants")
sys.path.insert(0, ROOT)


def build(specs):
    from twixt_for_open_spiel_b200 import build as b
    os.makedirs(VDIR, exist_ok=True)
    for spec in specs:
        name, _, flags = spec.partition("=")
        out = os.path.join(VDIR, name + ".so")
        b.build(out=out, extra_flags=[f for f in flags.split(",") if f])
        print("built", out)


def child(sizes, envs, reps):
    for n in sizes:
        child_one(n, envs, reps)


def child_one(n, envs, reps):
    import numpy as np
    import torch
    from oracle import pyoracle
    from twixt_for_open_spiel_b200 import TwixTBatch
    seed = 0x7477697854
    og = pyoracle.OracleGame(n)
    b = TwixTBatch(n, 96, 0, seed)
    rets, lens, _ = b.playout()
    recs = b.export_state()
    bad = 0
    for e in range(96):
        st = og.new_initial_state()
        acts = st.playout_philox(seed, e)
        bad += len(acts) != lens[e] or not np.array_equal(recs[e], st.export_record())
    b.close()
    b = TwixTBatch(n, envs, 0, seed)
    b.use_torch_stream()
    ms = []
    plies = 0
    for i in range(reps + 2):
        b.set_seed(seed + i)
        b.reset()
        b.stats_reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.playout(want_returns=False, want_lengths=False)
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            ms.append(e0.elapsed_time(e1))
            plies = b.stats()["plies"]
    ms.sort()
    print("RESULT n=%d mismatches=%d min=%.3f ms median=%.3f ms  plies/launch=%d  %.2f G steps/s (median)" % (
        n, bad, ms[0], ms[len(ms) // 2], plies, plies / ms[len(ms) // 2] / 1e6))


def child_kernels():
    """the per-call kernels (bench.py's kernel section) with the library of this process"""
    import json
    import torch
    import bench
    from twixt_for_open_spiel_b200 import TwixTBatch
    peak, _ = bench._peaks()
    res = bench.kernel_microbench(torch, TwixTBatch, 24, 0, peak)
    print("RESULT " + json.dumps({k: {"ms": round(v["ms"], 4), "frac": round(v.get("frac", 0.0), 4)} for k, v in res.items()}))


def run_kernels():
    names = ["<product>"] + sorted(f for f in os.listdir(VDIR) if f.endswith(".so"))
    for rnd in range(2):
        for name in names:
            env = dict(os.environ)
            if name != "<product>":
                env["TWIXT_B200_LIB"] = os.path.join(VDIR, name)
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "child_kernels"], capture_output=True,
                                 text=True, env=env)
            line = [l for l in res.stdout.splitlines() if l.startswith("RESULT")]
            print("%-24s round %d  %s" % (name, rnd, line[0] if line else "FAILED: " + res.stderr[-600:]), flush=True)


def run(sizes, envs, reps, rounds):
    names = sorted(f for f in os.listdir(VDIR) if f.endswith(".so"))
    for rnd in range(rounds):  # several rounds, so that a drifting clock shows up as a difference between rounds
        for name in names:
            env = dict(os.environ, TWIXT_B200_LIB=os.path.join(VDIR, name))
            try:
                res = subprocess.run([sys.executable, os.path.abspath(__file__), "child", sizes, str(envs), str(reps)],
                                     capture_output=True, text=True, env=env, timeout=150 * len(sizes.split(",")))
            except subprocess.TimeoutExpired:
                print("%-28s round %d  TIMEOUT (hung kernel?)" % (name, rnd), flush=True)
                return
            lines = [l for l in res.stdout.splitlines() if l.startswith("RESULT")]
            for line in lines or ["FAILED: " + res.stderr[-400:]]:
                print("%-28s round %d  %s" % (name, rnd, line), flush=True)
            if res.returncode != 0 and lines:
                print("%-28s round %d  FAILED: %s" % (name, rnd, res.stderr[-400:]), flush=True)


if __name__ == "__main__":
    if sys.argv[1] == "build":
        build(sys.argv[2:])
    elif sys.argv[1] == "child_kernels":
        child_kernels()
    elif sys.argv[1] == "kernels":
        run_kernels()
    elif sys.argv[1] == "child":
        child([int(x) for x in sys.argv[2].split(",")], int(sys.argv[3]), int(sys.argv[4]))
    else:
        a = sys.argv[2:]
        run(a[0] if a else "24", int(a[1]) if len(a) > 1 else 1 << 20, int(a[2]) if len(a) > 2 else 5,
            int(a[3]) if len(a) > 3 else 2)
