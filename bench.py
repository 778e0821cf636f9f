#!/usr/bin/env python3
"""bench.py -- headline benchmark: env steps/sec of fused random playouts,
twixt(board_size=24), 1 Mi envs per GPU (BASELINE.json configs[3]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch: every env of the rank's
shard is reset to the initial position and played to a terminal state with
uniformly random legal moves (Philox stream per global env id, so results do
not depend on the GPU count).  Envs shard across ranks with no data-path
collective; the only exchange is the final reduction of the counters.

Prints ONE JSON line (see the key list in the task contract):
  value      whole-job plies / max-over-ranks device time, state resident in HBM
  e2e        the same metric through the C ABI with HOST (pinned) buffers:
             per step the per-env stream ids go host->device and returns +
             lengths come device->host inside the timed region
  roofline   the fused playout kernel against its PHYSICAL ceiling, the issue slots
             of the device (148 SMs x 4 schedulers x f_SM x 32 lanes / thread-
             instructions per ply, the latter from the committed ncu capture of
             this build, profiles/r2_playout_ncu.json); the algorithmic-bytes
             convention of SURVEY.md section 8(d) (2*S(24) = 1328 B per env-step
             against the measured HBM peak) is kept beside it as `hbm_convention`
  configs    the other BASELINE.json configs that are benchmarks: c1_n8 (1 Mi-env
             playouts at n=8) and c3_n12 (4 096 MCTS leaves x 4 rollouts), each
             with the reference's CPU path timed beside it
  adapter_latency_us   per-call cost of the single-state calls a drop-in adapter
             makes (count = 1, host buffers), beside the reference's own ns
  cpu_baseline  the reference's own CPU path (oracle/_ref/ref_bench: unmodified
             reference sources) on this host's cores, bounded sample
`--impl reference` times only that CPU path, as the reference arm.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 0x7477697854  # "twixT"
METRIC = "env_steps_per_sec_random_playouts_board24"
UNIT = "steps/s"
ALGO_BYTES_PER_STEP = 1328  # 2 * S(24), SURVEY.md section 8(d)
DUMP_BYTES_MAX = 64 * 10**6 - 4096  # --dump-outputs in all, less room for the .npy headers


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def _playout_capture():
    """Counters of the playout kernel from the committed `ncu --set full` capture of THIS build
    (tools/ncu_playout_json.py writes it from the .ncu-rep): warp instructions, active lanes, issue-active,
    ALU pipe, DRAM bytes -- all per launch of the bench's own workload."""
    path = os.path.join(ROOT, "profiles", "r2_playout_ncu.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def _host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference(board_size: int, seconds: float, mode: str = "clone"):
    """The reference's CPU playout loop on all host cores (one process per core)."""
    from oracle import pyoracle
    cores = _host_cores()
    res = pyoracle.run_ref_bench(board_size, cores, seconds, mode)
    if res is not None:
        return res["steps_per_sec"], "reference", cores, res
    # oracle/_ref absent (reference tree was never available to build it): time the C port
    import multiprocessing as mp
    with mp.get_context("fork").Pool(cores) as pool:
        t0 = time.time()
        outs = pool.starmap(_port_worker, [(board_size, seconds, 1 + i) for i in range(cores)])
        wall = time.time() - t0
    plies = sum(o[0] for o in outs)
    el = max(o[2] for o in outs)
    return plies / el, "port", cores, {"plies": plies, "games": sum(o[1] for o in outs), "seconds": el, "wall": wall}


def _port_worker(board_size, seconds, seed):
    import ctypes as C
    from oracle import pyoracle
    g = pyoracle.OracleGame(board_size)
    games, el = C.c_int64(0), C.c_double(0)
    plies = pyoracle.oracle_lib().oracle_bench_playouts(g.h, seconds, seed, C.byref(games), C.byref(el))
    return int(plies), int(games.value), float(el.value)


def cpu_reference_raw(board_size: int, workers: int, seconds: float, mode: str):
    """oracle/_ref/ref_bench in one of its other modes ("rollout", "latency"); None if it is not built."""
    from oracle import pyoracle
    return pyoracle.run_ref_bench(board_size, workers, seconds, mode)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    per_step = args.ref_seconds
    for _ in range(args.warmup):
        cpu_reference(args.board_size, min(per_step, 1.0))
    vals, detail, kind, cores = [], None, "reference", _host_cores()
    t0 = time.time()
    for _ in range(args.steps):
        v, kind, cores, detail = cpu_reference(args.board_size, per_step)
        vals.append(v)
    wall = time.time() - t0
    value = sum(vals) / len(vals)
    faithful = None
    try:
        faithful, _, _, _ = cpu_reference(args.board_size, min(3.0, per_step), "faithful")
    except Exception:
        pass
    sample = ("%d steps x %.1f s of random playouts from the initial position on %d processes, one prebuilt "
              "initial state per process + Clone() per game (steel-man; the reference's own NewInitialState-per-game "
              "path is 'faithful_value')" % (args.steps, per_step, cores))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "twixt(board_size=%d) random playouts, reference CPU path (oracle/_ref/ref_bench)"
                   % args.board_size, "board_size": args.board_size},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                         "faithful_value": faithful},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def kernel_microbench(torch, TwixTBatch, board_size, device, peak_gbs):
    """Per-kernel roofline lines for K1 (legal list/mask), K2+K3 (apply) and K4 (observation)
    on mid-game states; algorithmic bytes per unit from SURVEY.md section 8(d)."""
    out = {}
    n = board_size
    S = 9 * ((n * n + 7) // 8) + 16
    E = 1 << 20
    b = TwixTBatch(n, E, device, SEED)
    b.use_torch_stream()
    b.playout(max_plies=200, want_returns=False, want_lengths=False)
    dev = torch.device("cuda", device)

    def timed(fn, reps=5):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for s, e in evs:
            s.record()
            fn()
            e.record()
        torch.cuda.synchronize(dev)
        return min(s.elapsed_time(e) for s, e in evs) * 1e-3

    acts = torch.zeros((E, b.max_legal_actions), dtype=torch.int16, device=dev)
    cnts = torch.zeros(E, dtype=torch.int32, device=dev)
    t = timed(lambda: b.legal_actions(out_actions=acts, out_counts=cnts))
    mean_l = float(cnts.float().mean().item())
    bytes_unit = (2 * ((n * n + 7) // 8) + 16) + 4 + 2 * mean_l
    out["legal_list"] = {"envs_per_s": E / t, "ms": t * 1e3, "algo_bytes_per_env": bytes_unit,
                         "achieved_gbs": E * bytes_unit / t / 1e9, "frac": E * bytes_unit / t / 1e9 / peak_gbs}
    # the same list as int64 (open_spiel::Action), what a drop-in LegalActions() binding asks for
    acts64 = torch.zeros((E, b.max_legal_actions), dtype=torch.int64, device=dev)
    t = timed(lambda: b.legal_actions(out_actions=acts64, out_counts=cnts))
    bytes_unit = (2 * ((n * n + 7) // 8) + 16) + 4 + 8 * mean_l
    out["legal_list_i64"] = {"envs_per_s": E / t, "ms": t * 1e3, "algo_bytes_per_env": bytes_unit,
                             "achieved_gbs": E * bytes_unit / t / 1e9, "frac": E * bytes_unit / t / 1e9 / peak_gbs}
    del acts64
    mask = torch.zeros((E, n * n), dtype=torch.uint8, device=dev)
    t = timed(lambda: b.legal_mask(out=mask))
    bytes_unit = (2 * ((n * n + 7) // 8) + 16) + n * n
    out["legal_mask"] = {"envs_per_s": E / t, "ms": t * 1e3, "algo_bytes_per_env": bytes_unit,
                         "achieved_gbs": E * bytes_unit / t / 1e9, "frac": E * bytes_unit / t / 1e9 / peak_gbs}
    # apply: one random legal move per env (a random entry of its legal list), statuses on device; the records
    # are restored from a device snapshot BEFORE each timed launch, and only the apply launch is bracketed
    idx = (torch.rand(E, device=dev) * cnts.clamp(min=1).float()).long().clamp(max=b.max_legal_actions - 1)
    move = acts.gather(1, idx.view(-1, 1)).view(-1).to(torch.int32)
    move = torch.where(cnts > 0, move, torch.full_like(move, -1))
    status = torch.zeros(E, dtype=torch.int32, device=dev)
    snap = torch.empty((E, b.record_words), dtype=torch.int32, device=dev)
    b.export_state(out=snap)
    b.set_validation(False)  # our own export: a plain device copy
    ts = []
    for rep in range(7):
        b.import_state(snap)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.apply(move, out_status=status)
        e1.record()
        torch.cuda.synchronize(dev)
        if rep >= 2:
            ts.append(e0.elapsed_time(e1) * 1e-3)
    b.set_validation(True)
    t = min(ts)
    out["apply"] = {"steps_per_s": E / t, "ms": t * 1e3, "algo_bytes_per_step": 2 * S,
                    "achieved_gbs": E * 2 * S / t / 1e9, "frac": E * 2 * S / t / 1e9 / peak_gbs,
                    "illegal": int((status == 1).sum().item()), "timing": "CUDA events around the apply launch only"}
    # import validation: one streaming pass over the records (validate kernel) + the device copy
    t_val = timed(lambda: b.import_state(snap))
    out["import_validated"] = {"envs_per_s": E / t_val, "ms": t_val * 1e3,
                               "note": "validate kernel + device-to-device copy + 8-byte verdict read back"}
    b.close()
    del acts, mask, snap
    E4 = 1 << 16
    b = TwixTBatch(n, E4, device, SEED)
    b.use_torch_stream()
    b.playout(max_plies=200, want_returns=False, want_lengths=False)
    obs = torch.empty((E4,) + b.obs_shape, dtype=torch.float32, device=dev)
    t = timed(lambda: b.observation(out=obs))
    bytes_unit = S + 48 * n * (n - 2)
    out["observation"] = {"envs_per_s": E4 / t, "ms": t * 1e3, "algo_bytes_per_env": bytes_unit,
                          "achieved_gbs": E4 * bytes_unit / t / 1e9, "frac": E4 * bytes_unit / t / 1e9 / peak_gbs}
    # BASELINE config C5: B = 65 536 mid-game states -> [B,12,n,n-2] f32 + [B,n*n] u8 by ONE launch
    # (twixt_observation_and_mask through the torch / DLPack producer)
    from twixt_for_open_spiel_b200.producer import ObservationMaskProducer
    prod = ObservationMaskProducer(b)
    t = timed(lambda: prod.produce())
    bytes_unit = S + 48 * n * (n - 2) + n * n
    out["obs_mask"] = {"envs_per_s": E4 / t, "ms": t * 1e3, "algo_bytes_per_env": bytes_unit, "batch": E4,
                       "achieved_gbs": E4 * bytes_unit / t / 1e9, "frac": E4 * bytes_unit / t / 1e9 / peak_gbs,
                       "workload": "BASELINE configs[4]: %d mid-game states, obs + legal mask in one pass" % E4}
    del prod
    b.close()
    return out


def other_configs(torch, TwixTBatch, device, args):
    """BASELINE.json configs[0] (n = 8 playouts, the reference's default) and configs[2] (n = 12 MCTS leaf
    rollouts, rollout_count = 4), each with the reference's CPU path on this host beside it."""
    import numpy as np
    from twixt_for_open_spiel_b200.rollout import BatchedRolloutEvaluator
    dev = torch.device("cuda", device)
    cores = _host_cores()
    out = {}
    # ---- C1: 1 Mi-env random playouts at n = 8
    n, E = 8, 1 << 20
    b = TwixTBatch(n, E, device, SEED)
    b.use_torch_stream()
    rets = torch.zeros((E, 2), dtype=torch.float32, device=dev)
    lens = torch.zeros(E, dtype=torch.int32, device=dev)
    ms = []
    for i in range(3 + 5):
        b.set_seed(SEED + i)
        b.reset()
        b.stats_reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.playout(out_returns=rets, out_lengths=lens)
        e1.record()
        torch.cuda.synchronize(dev)
        if i >= 3:
            ms.append(e0.elapsed_time(e1))
    plies = b.stats()["plies"]
    ids = np.arange(E, dtype=np.uint64)
    rets_h, lens_h = np.zeros((E, 2), dtype=np.float32), np.zeros(E, dtype=np.int32)
    b.reset()
    b.playout(stream_ids=ids, out_returns=rets_h, out_lengths=lens_h)
    t0 = time.perf_counter()
    e2e_plies = 0
    for i in range(3):
        b.set_seed(SEED + 100 + i)
        b.reset()
        b.playout(stream_ids=ids, out_returns=rets_h, out_lengths=lens_h)
        e2e_plies += int(lens_h.sum())
    e2e_s = time.perf_counter() - t0
    b.close()
    med = statistics.median(ms)
    c1 = {"workload": "twixt(board_size=8) %d-env random playouts to terminal (BASELINE.json configs[0])" % E,
          "value": plies / (med * 1e-3), "unit": UNIT, "ms_per_launch": med, "plies_per_launch": plies,
          "e2e": {"value": e2e_plies / e2e_s, "unit": UNIT, "h2d_bytes_per_step": E * 8, "d2h_bytes_per_step": E * 12}}
    ref = None if args.no_cpu else cpu_reference_raw(8, cores, 3.0, "clone")
    if ref is not None:
        c1["cpu_baseline"] = {"value": ref["steps_per_sec"], "unit": UNIT, "cores": cores, "kind": "reference",
                              "sample": "3 s of n=8 random playouts, %d processes, Clone() per game" % cores}
    out["c1_n8"] = c1
    # ---- C3: 4 096 leaves at a random ply in [0, 60] x 4 rollouts, n = 12
    n, B, R = 12, 4096, 4
    ev = BatchedRolloutEvaluator(n, n_rollouts=R, max_leaves=B, device=device, seed=SEED)
    eb = ev.batch
    for d in range(61):  # leaf e sits at ply ~ e*61/B: contiguous ranges of equal depth, made on the device
        lo, hi = (d * B + 60) // 61, ((d + 1) * B + 60) // 61
        if hi > lo and d > 0:
            eb.playout(lo, hi - lo, max_plies=d, want_returns=False, want_lengths=False)
    leaves = eb.export_state(0, B)
    ev.evaluate_records(leaves)  # warm-up (staging buffers)
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        host_means = ev.evaluate_records(leaves)
    t_host = (time.perf_counter() - t0) / reps
    eb.set_validation(False)
    t0 = time.perf_counter()
    for _ in range(reps):
        ev.evaluate_records(leaves)
    t_trusted = (time.perf_counter() - t0) / reps
    eb.set_validation(True)
    eb.import_state(leaves, 0)
    ev.evaluate_slots(B)  # warm-up
    t0 = time.perf_counter()
    for _ in range(reps):
        dev_means = ev.evaluate_slots(B)
    t_dev = (time.perf_counter() - t0) / reps
    rec_bytes = int(leaves.nbytes)
    c3 = {"workload": "twixt(board_size=12) %d MCTS leaves (ply 0..60) x %d random rollouts each, mean returns per leaf "
                      "(BASELINE.json configs[2], mcts_example --rollout_count=4 shape)" % (B, R),
          "value": B / t_host, "unit": "leaves/s", "rollouts_per_s": B * R / t_host, "ms_per_batch": t_host * 1e3,
          "api": "BatchedRolloutEvaluator.evaluate_records(host records): validated import, device clone x4, ONE "
                 "playout launch, returns to the host",
          "h2d_bytes_per_batch": rec_bytes + B * R * 16, "d2h_bytes_per_batch": B * R * 8,
          "trusted_import": {"value": B / t_trusted, "unit": "leaves/s", "ms_per_batch": t_trusted * 1e3},
          "device_resident": {"value": B / t_dev, "unit": "leaves/s", "ms_per_batch": t_dev * 1e3,
                              "api": "evaluate_slots: leaves already in env slots on the device; clone, playout and "
                                     "the mean stay on the device", "h2d_bytes_per_batch": 0,
                              "d2h_bytes_per_batch": B * 8},
          "mean_abs_return": float(np.abs(host_means).mean()), "device_mean_abs_return": float(np.abs(dev_means).mean())}
    ref = None if args.no_cpu else cpu_reference_raw(12, cores, 3.0, "rollout")
    if ref is not None:
        c3["cpu_baseline"] = {"value": ref["leaves_per_sec"], "unit": "leaves/s", "cores": cores, "kind": "reference",
                              "sample": "3 s of the reference's rollout evaluation (4 x Clone + random playout per "
                                        "leaf), %d processes" % cores}
    ev.close()
    out["c3_n12"] = c3
    return out


def adapter_latency(TwixTBatch, n, device, args):
    """What ONE State method costs through the C ABI with count = 1 and host buffers (kernel launch +
    synchronise; small host transfers go through the pinned, device-mapped arena), i.e. the per-call price an
    unbatched open_spiel driver pays, beside the reference's own per-call time on this host
    (oracle/_ref/ref_bench latency).  The adapters do not make the four query calls per move: they call
    twixt_step once per ApplyAction and keep its answer (`step_apply_and_query`)."""
    import numpy as np
    b = TwixTBatch(n, 8, device, SEED)
    b.playout(0, 8, max_plies=150, want_returns=False, want_lengths=False)
    acts = np.zeros((1, b.max_legal_actions), dtype=np.int64)
    cnt = np.zeros(1, dtype=np.int32)
    obs = np.zeros((1,) + b.obs_shape, dtype=np.float32)
    term = np.zeros(1, dtype=np.uint8)
    ret = np.zeros((1, 2), dtype=np.float32)

    def per_call(fn, reps=400):
        for _ in range(20):
            fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t0) / reps * 1e6

    res = {"board_size": n, "count": 1, "buffers": "host (pageable numpy)", "unit": "us per call",
           "note": "through ctypes (about 1 us of the figure is the Python call itself)"}
    res["legal_actions"] = per_call(lambda: b.legal_actions(0, 1, out_actions=acts, out_counts=cnt))
    res["observation_tensor"] = per_call(lambda: b.observation(0, 1, out=obs))
    res["is_terminal"] = per_call(lambda: b.is_terminal(0, 1, out=term))
    res["returns"] = per_call(lambda: b.returns(0, 1, out=ret))
    res["clone"] = per_call(lambda: b.clone(0, 1, 1))
    # apply: a legal move each time (the state is restored by a device clone outside the timed call)
    b.clone(0, 2, 1)
    b.legal_actions(0, 1, out_actions=acts, out_counts=cnt)
    move = np.array([acts[0, 0]], dtype=np.int32)
    status = np.zeros(1, dtype=np.int32)
    tot = 0.0
    for i in range(220):
        b.clone(2, 0, 1)
        b.synchronize()
        t0 = time.perf_counter()
        b.apply(move, 0, out_status=status)
        if i >= 20:
            tot += time.perf_counter() - t0
    res["apply_action"] = tot / 200 * 1e6
    # twixt_step: ApplyAction + IsTerminal + CurrentPlayer + Returns + LegalActions of the new state in ONE launch
    # (what the adapters call per move; the four queries are then served from the host)
    legal = np.empty(b.max_legal_actions, dtype=np.int64)
    tot = 0.0
    for i in range(220):
        b.clone(2, 0, 1)
        b.synchronize()
        t0 = time.perf_counter()
        b.step(0, int(move[0]), out_legal=legal)
        if i >= 20:
            tot += time.perf_counter() - t0
    res["step_apply_and_query"] = tot / 200 * 1e6
    b.close()
    ref = None if args.no_cpu else cpu_reference_raw(n, 1, 1.5, "latency")
    if ref is not None:
        res["reference_ns"] = {k: ref[k] for k in ("legal_actions_ns", "apply_action_ns", "observation_tensor_ns",
                                                   "clone_ns", "is_terminal_returns_ns")}
    return res


def dump_outputs(out_dir, outputs, suffix=""):
    """Writes what the timed playout handed back in its last step as float32 `<name><suffix>.npy`: `returns`
    [E, 2] and `lengths` [E] (plies per game, exact in float32).  Seeds and stream ids depend only on the
    arguments, so two builds run with the same arguments can be compared array for array.  Above
    DUMP_BYTES_MAX the same seeded sample of envs is taken from every array and its indices go to `env_index`."""
    import numpy as np
    arrays = {name: t.cpu().numpy().astype(np.float32) for name, t in outputs.items()}
    envs = len(next(iter(arrays.values())))
    per_env = sum(a[0].nbytes for a in arrays.values())
    if envs * per_env > DUMP_BYTES_MAX:
        keep = DUMP_BYTES_MAX // (per_env + 8)
        idx = np.sort(np.random.default_rng(SEED).choice(envs, size=keep, replace=False))
        arrays = {name: a[idx] for name, a in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from twixt_for_open_spiel_b200 import TwixTBatch
    from twixt_for_open_spiel_b200.sharding import reduce_counters, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    n, E = args.board_size, args.envs
    batch = TwixTBatch(n, E, local, SEED)
    batch.use_torch_stream()
    first_id, _ = shard_range(E * world, world, rank)  # weak scaling: E envs per GPU
    batch.set_stream_base(first_id)  # global env ids: shard r owns [r*E, (r+1)*E)
    rets = torch.zeros((E, 2), dtype=torch.float32, device=dev)
    lens = torch.zeros(E, dtype=torch.int32, device=dev)

    def step(i):
        batch.set_seed(SEED + i)
        batch.reset()
        batch.playout(out_returns=rets, out_lengths=lens)

    for i in range(args.warmup):
        step(i)
    barrier()
    batch.stats_reset()
    launches0 = batch.stats()["kernel_launches"]
    k_evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    ev0.record()
    for i in range(args.steps):
        batch.set_seed(SEED + args.warmup + i)
        batch.reset()
        k_evs[i][0].record()
        batch.playout(out_returns=rets, out_lengths=lens)
        k_evs[i][1].record()
    ev1.record()
    barrier()
    clocks = sampler.stop()
    elapsed_ms = ev0.elapsed_time(ev1)
    st = batch.stats()
    launches = st["kernel_launches"] - launches0
    kernel_ms = [s.elapsed_time(e) for s, e in k_evs]

    tot = reduce_counters(st, dist if world > 1 else None, dev)  # the only collective of the whole job
    tmax = torch.tensor([elapsed_ms, sum(kernel_ms) / len(kernel_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    red = [tot["plies"], tot["games"], tot["red_wins"], tot["blue_wins"], tot["draws"], tot["swaps"]]
    total_plies = int(red[0])
    elapsed_s = float(tmax[0].item()) * 1e-3
    value = total_plies / elapsed_s
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"returns": rets, "lengths": lens}, "_rank%d" % rank if world > 1 else "")

    # ---- e2e: the same workload through the C ABI with HOST buffers -------------
    ids_host = torch.arange(rank * E, (rank + 1) * E, dtype=torch.int64).pin_memory()
    rets_host = torch.zeros((E, 2), dtype=torch.float32).pin_memory()
    lens_host = torch.zeros(E, dtype=torch.int32).pin_memory()
    ids_np = ids_host.numpy().view(np.uint64)
    rets_np, lens_np = rets_host.numpy(), lens_host.numpy()
    e2e_steps = args.steps  # the same number of steps as the device-timed arm

    def e2e_step(i):
        batch.set_seed(SEED + 1000 + i)
        batch.reset()
        batch.playout(stream_ids=ids_np, out_returns=rets_np, out_lengths=lens_np)  # H2D ids, D2H results, sync
        return int(lens_np.sum())

    e2e_step(-1)
    barrier()
    t0 = time.perf_counter()
    e2e_plies = 0
    for i in range(e2e_steps):
        e2e_plies += e2e_step(i)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_red = torch.tensor([e2e_plies], dtype=torch.int64, device=dev)
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_red, op=dist.ReduceOp.SUM)
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = int(e2e_red.item()) / float(e2e_t.item())

    if rank == 0:
        peak, peak_src = _peaks()
        plies_per_launch = st["plies"] / args.steps
        k_ms = sum(kernel_ms) / len(kernel_ms)
        kernel_steps_per_s = plies_per_launch / (k_ms * 1e-3)
        conv = plies_per_launch * ALGO_BYTES_PER_STEP / (k_ms * 1e-3) / 1e9
        cap = _playout_capture()
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        f_sm = 1e6 * float(clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965)
        roofline = {
            "bound": "issue", "kernel": "playout_kernel<24>", "unit": "steps/s", "achieved": kernel_steps_per_s,
            "kernel_ms": k_ms, "kernel_ms_median": statistics.median(kernel_ms), "kernel_ms_best": min(kernel_ms),
            "steps_per_launch": plies_per_launch,
            "ceiling": "SMs x 4 schedulers x f_SM x 32 lanes / thread-instructions per ply: every issue slot used, "
                       "every lane active, at this build's instruction count",
            # what the HBM convention of SURVEY 8(d) gives for the same launch (state streamed once per MOVE;
            # the kernel streams it once per GAME, so this is not a physical fraction)
            "hbm_convention": {"achieved_gbs": conv, "peak_gbs": peak, "frac": conv / peak,
                               "algorithmic_bytes_per_step": ALGO_BYTES_PER_STEP, "peak_source": peak_src},
        }
        if cap is not None:
            tipp = cap["thread_inst_per_launch"] / cap["plies_per_launch"]
            ceiling = sms * 4 * f_sm * 32 / tipp
            roofline.update({
                "peak": ceiling, "frac": kernel_steps_per_s / ceiling, "thread_inst_per_ply": tipp,
                "sm_count": sms, "f_sm_hz": f_sm,
                "traffic": cap["dram_bytes_per_launch"],
                "dram_frac_of_measured_peak": cap["dram_bytes_per_launch"] / (k_ms * 1e-3) / 1e9 / peak,
                "ncu": {k: cap[k] for k in ("source", "warp_inst_per_launch", "lanes_per_warp_inst", "issue_active_pct",
                                            "alu_pipe_pct", "fma_pipe_pct", "lsu_pipe_pct", "warps_per_sm",
                                            "registers", "duration_ms") if k in cap},
            })
        else:
            roofline.update({"peak": None, "frac": None, "traffic": None,
                             "note": "profiles/r2_playout_ncu.json (ncu capture of this build) is missing"})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_s * 1e3 / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "twixt(board_size=%d) %d-env random playouts per GPU to terminal "
                                   "(BASELINE.json configs[3])" % (n, E),
                       "board_size": n, "envs_per_gpu": E, "global_envs": E * world,
                       "parallelism": "envs sharded x%d, no data-path collective" % world,
                       "l2": "inputs larger than L2: %.0f MB of env records per GPU vs 126 MB L2"
                             % (E * batch.record_words * 4 / 1e6),
                       "rng": "Philox4x32-10, key=seed+step, stream=global env id"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(ids_host.numel() * 8),
                    "d2h_bytes_per_step": int(rets_host.numel() * 4 + lens_host.numel() * 4),
                    "steps": e2e_steps, "api": "twixt_reset + twixt_playout(host stream_ids, host returns/lengths)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "outcomes": {"plies": total_plies, "games": int(red[1]), "red": int(red[2]), "blue": int(red[3]),
                         "draws": int(red[4]), "swaps": int(red[5]), "max_length": int(tot["max_length"])},
        }
        if world == 1 and not args.no_cpu:
            v, kind, cores, detail = cpu_reference(n, args.cpu_seconds)
            faithful = None
            if kind == "reference":
                faithful = cpu_reference(n, min(5.0, args.cpu_seconds), "faithful")[0]
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": cores, "kind": kind,
                "sample": "%.0f s of random playouts from the initial position, %d processes, Clone() of a prebuilt "
                          "initial state per game (steel-man); faithful_value = NewInitialState() per game as the "
                          "reference example does" % (args.cpu_seconds, cores),
                "faithful_value": faithful}
        if world == 1 and not args.no_kernels:
            line["kernels"] = kernel_microbench(torch, TwixTBatch, n, local, peak)
        if world == 1 and not args.no_configs:
            line["configs"] = other_configs(torch, TwixTBatch, local, args)
            line["adapter_latency_us"] = adapter_latency(TwixTBatch, n, local, args)
        print(json.dumps(line))
    batch.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--board-size", type=int, default=24)
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--ref-seconds", type=float, default=3.0, help="CPU sample per step of the reference arm")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-kernels", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip configs c1_n8 / c3_n12 and adapter_latency_us")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's returns and lengths to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
