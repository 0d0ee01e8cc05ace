#!/usr/bin/env python
"""bench.py -- switch-agent decisions/sec of the SwitchFL lockstep hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA, one rank per GPU under torchrun)
    python bench.py --impl reference [...]                         the reference's CPU path (oracle port, all host cores)

Headline workload: BASELINE.json configs[3], the configuration the north-star target is quoted on -- the large synthetic map
(100x100, 50 trains, 354 switches, malfunctions 0.01 / 5-15; ``c4_rail100_t50``) with 8192 lockstep environments per GPU
(65536 on 8), every environment an independent distributed-Q learner (gamma 1, eps .5 decay .9997, lr .1).  One "step" =
one launch of the hot-path kernel advancing every environment by ``--ticks`` flatland ticks plus every switch-agent
decision, Q-update and episode reset in between.  N > 1: the same per GPU (weak scaling), environments sharded by seed
range, no data-path collective (SURVEY.md section 8e).  The other configurations (C2 = configs[1], C3 = configs[2],
C5 = configs[4]) are measured in the same run and reported under ``extra``.

Prints ONE JSON line (rank 0).  value = device-timed (CUDA events on the launch stream, max over ranks) decisions/s with
all state resident in HBM; e2e = the same metric through the public drop-in API the reference's scripts call --
``DistrQLearning.learn(num_episodes, ...)`` (main.py:63) -- wall clock, with the per-env hyper-parameter block copied
host->device and the per-env counters / episode logs copied device->host inside the timed region.

``--dump-outputs DIR`` writes what the headline workload's environments hold after the last timed step (rank 0) as
float64 ``DIR/<name>.npy`` files, so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                                            # the benchmark leaves the source tree as it found it
from __graft_entry__ import load_package  # noqa: E402

METRIC = "switch_agent_decisions_per_sec"
HP = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)   # test_model.py:56-63
SEED = 450565
C3_SEEDS = (64, 65, 66, 67, 69)                                          # hyperparam_tuning.py:10
# workload -> (fixture, envs per GPU, Q hash rows per env, description); "@c3" = the five seed maps of the hyper-parameter grid
WORKLOADS = {
    "c2": ("c1_synth18", 4096, 1024,
           "C2: 4096 lockstep envs of the test_model.py map (18x18, 2 trains, malfunctions; c1_synth18 stand-in), distributed Q-learning, learn mode"),
    "c3": ("@c3", 20480, 32768,
           "C3: hyperparam_tuning.py default grid (eps .5, decay .9997, lr .1) x seeds {64,65,66,67,69} = 5 maps (80x80, 15 trains, "
           "25 cities, double track, no malfunctions; synthetic stand-ins), each (map, point) replicated with distinct RNG streams: "
           "5 x 4096 envs per GPU, distributed Q-learning, learn mode"),
    "c4": ("c4_rail100_t50", 8192, 65536,
           "C4: large synthetic map (100x100, 50 trains, 354 switches, double track, malfunctions 0.01 / 5-15), 65536 envs per "
           "8 GPUs = 8192 per GPU, distributed Q-learning, learn mode"),
    "c5": ("c4_rail100_t50", 8192, 2,
           "C5 (extension, no reference counterpart): the C4 map in shared-table mode -- all 8192 envs of a GPU read one dense "
           "Q table and accumulate TD steps; every step the integer accumulators are all-reduced over the GPUs (NCCL) and the "
           "mean step is folded into the table"),
}
TICKS = {"c2": 8192, "c3": 1024, "c4": 1024, "c5": 1024}                 # flatland ticks per env per step (launch)
FIXTURE = None                                                            # set in main (the CPU workers re-derive the maps from it)


def fixture_path(name):
    return name if name.startswith("@") else os.path.join(ROOT, "tests", "golden", name + ".fixture.npz")


def workload_fixtures(fixture=None):
    """The maps of a workload: one for C2 / C4 / C5, the five seed maps of the hyper-parameter grid for C3."""
    from switchfl_b200 import mapgen
    fixture = fixture or FIXTURE
    if fixture == "@c3":                                                  # hyperparam_tuning.py:17-26, synthetic stand-ins
        return [mapgen.c3_fixture(s) for s in C3_SEEDS]
    return [mapgen.load_fixture(fixture)]


def bytes_per_decision(k_bar: float, P: float, A: float, A2: float) -> float:
    """Algorithmic bytes per decision, SURVEY.md section 8(d):  24*k + (26P+23) + 8A + (24P+138) + (32+8A')."""
    return 24.0 * k_bar + (26.0 * P + 23.0) + 8.0 * A + (24.0 * P + 138.0) + (32.0 + 8.0 * A2)


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampled every 20 ms for the whole run; the median SM clock is taken over the samples that fall inside
    the device-timed region of the headline workload."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.window = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def mark(self, t0, t1):
        self.window = (t0, t1)

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, sm_in, mx, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                clk, cmax = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            sm.append(clk); mx.append(cmax)
            inside = False
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                inside = bool(self.window and self.window[0] <= ts <= self.window[1])
            except ValueError:
                pass
            if inside:
                sm_in.append(clk)
            if inside or not self.window:
                for n, v in zip(names, parts[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        os.unlink(self.f.name)
        if sm:
            use = sm_in if sm_in else sm
            out.update(sm_mhz=float(np.median(use)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                       samples_in_timed_region=len(sm_in))
        return out


# ---------------------------------------------------------------------------------------------- CPU arm
def _cpu_worker(args):
    seed, budget_s, n_ep, fixture = args
    load_package()
    from switchfl_b200 import backend
    from oracle.switchfl_oracle import SwitchFLOracle
    fxs = workload_fixtures(fixture)
    fx = fxs[seed % len(fxs)]
    rm = backend.RailMap(fx)
    o = SwitchFLOracle(fx, rm.tab, seed=seed, **HP)
    rng = np.random.default_rng(seed)
    o.episode = 0
    t0 = time.perf_counter()
    dec = eps = 0
    while True:
        try:
            m = o.run_episode(rng, greedy=False, learn=True)
        except RuntimeError as ex:                         # the reference dies here too (observer.py:294-307): the run ends
            if "No train detected" not in str(ex):
                raise
            break
        dec += m["decisions"]
        eps += 1
        if (n_ep and eps >= n_ep) or (not n_ep and time.perf_counter() - t0 >= budget_s):
            break
    return dec, time.perf_counter() - t0, eps


def cpu_sample(budget_s: float, cores: int, n_ep: int = 0, seed0: int = SEED):
    """The reference's parallelism model (hyperparam_tuning.py:85-91): independent OS processes, one per core,
    one seed each, no communication; each runs the oracle's learn() episodes."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(seed0 + i, budget_s, n_ep, FIXTURE) for i in range(cores)])
    wall = time.perf_counter() - t0
    dec = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return dec, busy, wall, sum(r[2] for r in res)


CPU_NOTE = ("CPU oracle port of the reference path (the reference itself needs flatland, absent here); measured in the build container on "
            "one process, the port is 2-7x FASTER than the reference's own switchfl code on the same flatland shim (C1: 1307 vs 180, "
            "C3: 2495 vs 1284 decisions/s, identical decision counts), and the shim is lighter than real flatland: ratios against "
            "this arm are conservative")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step_s = 2.0
    for _ in range(min(args.warmup, 1)):
        cpu_sample(per_step_s, cores)
    dec, busy = 0, 0.0
    for _ in range(args.steps):
        d, b, _, _ = cpu_sample(per_step_s, cores)
        dec += d
        busy += b
    value = dec / busy
    sample = (f"{cores} processes x about {per_step_s:.0f} s of oracle learn() episodes per step on {os.path.basename(FIXTURE)}, one seed per "
              f"process (hyperparam_tuning.py:85-91); whole episodes, so a step can run over")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * busy / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload][3], "n_envs": cores, "note": CPU_NOTE},
            "cpu_baseline": {"value": value, "unit": "decisions/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------- our arm
class Ctx:
    """torch / torch.distributed handles of this rank."""

    def __init__(self):
        import torch
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = f"cuda:{self.local}"
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device(self.dev))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, times, counts):
        """MAX of the timings, SUM of the work counters over the ranks."""
        if self.dist is None:
            return [float(x) for x in times], [int(x) for x in counts]
        t = self.torch.tensor(list(times), device=self.dev, dtype=self.torch.float64)
        c = self.torch.tensor(list(counts), device=self.dev, dtype=self.torch.int64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        self.dist.all_reduce(c, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()], [int(x) for x in c.tolist()]


def engine_kwargs(parts: int) -> dict:
    """Scheduling knobs bench.py passes to every Engine of a workload with ``parts`` maps: with several maps in flight at
    once the GPU is full, so the large-map kernel built for 7 CTAs per SM beats the 4-CTA ("roomy") build the library would
    pick for one such launch alone (C3: 4.41e8 against 4.03e8 decisions/s)."""
    return {"roomy": False} if parts > 1 else {}


def kernel_counters(workload):
    """Per-launch ncu counters of the workload's k_run (committed under profiles/, NOT measured by this run)."""
    path = os.path.join(ROOT, "profiles", "kernel_counters.json")
    if os.path.exists(path):
        return json.load(open(path)).get(workload)
    return None


DUMP_ENVS = 8192                                                          # environments whose counters / episode logs are dumped
DUMP_Q_ENVS = 16                                                          # environments whose Q tables are dumped
DUMP_Q_BYTES = 40 << 20                                                   # at most this much of Q rows (with the above: < 64 MB)


def _sample(n: int, k: int, salt: int) -> np.ndarray:
    """All of range(n) when n <= k, else k of them drawn with a fixed seed (the same indices in every run), sorted."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng([SEED, salt]).choice(n, k, replace=False))


def dump_outputs(out_dir: str, engs) -> None:
    """``--dump-outputs``: what a caller of the timed path reads back after its last step, one float64 .npy per array.

    env_index          the environments (concatenated over the maps) the per-env arrays cover
    counters_<field>   [env] the per-env counters (Engine.counters)
    ep_<field>         [env, ep_cap] the episode log (Engine.episode_log), ep_logged = episodes logged, ep_delays [env, ep_cap, T]
    q_env, q_key       [row] environment (shared-table mode: map) and state key of a Q row, rows sorted by (q_env, q_key)
    q_actions          [row] the number of actions of the row's switch
    q_val              [row, a_max] its action values, 0 beyond q_actions (every value written is finite)
    """
    cnt, logs = np.concatenate([eng.counters() for eng in engs]), [eng.episode_log() for eng in engs]
    envs = _sample(len(cnt), DUMP_ENVS, 0)
    out = {"env_index": envs}
    for k in ("decisions", "ticks", "train_ticks", "episodes", "err", "q_rows", "elapsed", "aborted", "forced_stops", "stop_actions",
              "arrived_trains"):
        out["counters_" + k] = cnt[k][envs]
    out["ep_logged"] = np.concatenate([n for n, _, _ in logs])[envs]
    ep = np.concatenate([log for _, log, _ in logs])[envs]
    for k in ("cum_reward", "decisions", "arrived", "num_malfunctions", "ticks"):
        out["ep_" + k] = ep[k]
    out["ep_delays"] = np.concatenate([d for _, _, d in logs])[envs]

    a_max = max(eng.sizes.a_max for eng in engs)                          # the maps of C3 differ

    def block(owner, eng, keys, vals):
        tab, NT = eng.map.tab, len(eng.map.trains.targets)
        n_act = tab.sw_A[tab.port_switch[keys.astype(np.int64) // (NT * 48)]]
        vals = np.pad(vals, ((0, 0), (0, a_max - vals.shape[1])))
        return np.full(len(keys), owner), keys, n_act, np.where(np.arange(a_max) < n_act[:, None], vals, 0.0)

    rows = []
    if engs[0].shared_q:
        for k, eng in enumerate(engs):
            q = eng.shared_q_table()
            rows.append(block(k, eng, np.arange(q.size // q.shape[-1]), q.reshape(-1, q.shape[-1])))
    else:
        Bp = engs[0].n_envs
        for g in _sample(Bp * len(engs), DUMP_Q_ENVS, 1):
            eng = engs[g // Bp]
            keys, vals = eng.q_rows(int(g % Bp))
            order = np.argsort(keys, kind="stable")
            rows.append(block(g, eng, keys[order], vals[order]))
    q_env, q_key, q_actions, q_val = (np.concatenate(x) for x in zip(*rows))
    keep = _sample(len(q_key), DUMP_Q_BYTES // (8 * (3 + q_val.shape[1])), 2)
    out.update(q_env=q_env[keep], q_key=q_key[keep], q_actions=q_actions[keep], q_val=q_val[keep])

    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def run_block(cx: Ctx, wl: str, args, steps: int, warmup: int, sampler=None, flush_l2="auto") -> dict:
    """Device-resident arm of one workload: Engine level, CUDA-event timed, one engine per map."""
    torch = cx.torch
    from switchfl_b200 import backend
    fixture, envs, q_cap, desc = WORKLOADS[wl]
    shared = wl == "c5"
    head = wl == args.workload
    ticks = (args.ticks if head else 0) or TICKS[wl]
    fxs = workload_fixtures(fixture_path(fixture))
    B = (args.envs if (args.envs and head) else envs)
    q_cap = args.q_cap if (args.q_cap and head) else q_cap
    parts = len(fxs)
    Bp = B // parts                                                       # environments per map
    B = Bp * parts
    kw = engine_kwargs(parts)
    if head:
        kw.update({"lanes": args.lanes or None, "cta_warps": args.cta_warps or None})
        if args.roomy >= 0:
            kw["roomy"] = bool(args.roomy)

    def seeds_of(k):
        return np.arange(Bp, dtype=np.uint64) + np.uint64(SEED + cx.rank * B + k * Bp)

    rms = [backend.RailMap(fx, device_bfs=cx.local) for fx in fxs]      # distance maps on the GPU (sfl_distance_map)
    engs = [backend.Engine(rm, n_envs=Bp, device=cx.dev, q_cap=q_cap, ep_cap=4, shared_q=shared, **kw) for rm in rms]
    for k, eng in enumerate(engs):
        eng.set_hparams(**HP, seeds=seeds_of(k), episodes=-1)
        eng.reset()
        eng.enable_q_init(True)
        if shared:
            eng.init_shared_q(HP["default_q"])
    sync_ev = []
    # Several maps (C3): one stream per engine, so that the launches of a step run concurrently -- a launch carries its map
    # as a kernel parameter, nothing is shared between contexts.  The step is bracketed on the current stream.
    streams = [torch.cuda.Stream(device=cx.dev) for _ in engs] if parts > 1 else None

    def launch_all(timed=False):
        if streams is None:
            for eng in engs:
                launch(eng, timed)
            return
        cur = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(cur)
        for eng, st in zip(engs, streams):
            st.wait_event(fork)
            with torch.cuda.stream(st):
                launch(eng, timed)
            join = torch.cuda.Event()
            join.record(st)
            cur.wait_event(join)

    def launch(eng, timed=False):
        if shared:
            # overlapped schedule: the integer all-reduce (NCCL) + apply of this step run on a second stream while the
            # next launch already reads the other table (Engine.run_shared)
            eng.run_shared(ticks, cx.dist)
        else:
            eng.run(backend.MODE_LEARN, ticks)

    # Timing hygiene: the env state + Q tables are larger than L2, but on the small map the lines a launch actually touches
    # are not (ncu: 11 MB of DRAM traffic per launch), so L2 is flushed between the timed steps (256 MB written); the
    # flush sits inside the bracketed region, i.e. `value` pays for it.  Large-map workloads touch GBs per launch.
    state_bytes = sum(eng.sizes.state_bytes for eng in engs)
    flush = None
    if flush_l2 == "on" or (flush_l2 == "auto" and state_bytes < (1 << 30)):
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=cx.dev)
    for _ in range(warmup):
        launch_all()
    cx.barrier()

    def totals():
        out = np.zeros(8, np.int64)
        for eng in engs:
            c = eng.counters()
            out += [int(c[k].sum()) for k in ("decisions", "ticks", "train_ticks", "episodes", "aborted", "forced_stops", "stop_actions",
                                              "arrived_trains")]
        return out

    t0 = totals()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    cx.barrier()
    wall0 = time.time()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for a, b in evs:
        if flush is not None:
            flush.zero_()
        a.record()
        launch_all(timed=True)
        b.record()
    if shared:
        for eng in engs:
            eng.shared_q_flush()                                          # the last synchronisations end inside the timed region
    stop.record()
    cx.barrier()
    if sampler:
        sampler.mark(wall0, time.time())
    ms = start.elapsed_time(stop)
    step_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    sync_ms = 0.0
    if shared:                                                            # the synchronisation alone (not overlapped), for the record
        for i in range(4):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            engs[0].shared_q_sync(cx.dist)
            b.record()
            if i:
                sync_ev.append((a, b))
        torch.cuda.synchronize()
        sync_ms = float(np.mean([a.elapsed_time(b) for a, b in sync_ev]))
    kern_ms = step_ms / (1 if streams else parts)                         # mean duration of ONE k_run launch (concurrent maps: of the step)
    t1 = totals()
    if head and args.dump_outputs and cx.rank == 0:
        dump_outputs(args.dump_outputs, engs)
    q_rows_max, state_mb = 0, 0.0
    variant = engs[0].describe_launch(backend.MODE_LEARN)
    lanes = engs[0].lanes
    shared_cells = engs[0]._shared_cells() if shared else 0
    for eng in engs:
        # On congested maps the reference itself dies in observer.py:294-307 ("No train detected at active switch");
        # the kernel abandons such an episode and resets the env.  Every other error bit is fatal here.
        eng.check_errors(allow=backend.ERR_NO_TRAIN_AT_SWITCH)
        q_rows_max = max(q_rows_max, int(eng.counters()["q_rows"].max()))
        state_mb += eng.sizes.state_bytes / 1e6
        eng.close()
    flushed = flush is not None
    del engs, flush
    torch.cuda.empty_cache()
    (ms, kern_ms, sync_ms), d = cx.reduce([ms, kern_ms, sync_ms], list(t1 - t0))
    dec, n_ticks, train_ticks, episodes, aborted, forced, stops, arrived = d
    T = int(rms[0].trains.T)
    k_bar = train_ticks / max(dec, 1)
    P = float(np.mean(np.concatenate([rm.tab.sw_P for rm in rms]))); A = float(np.mean(np.concatenate([rm.tab.sw_A for rm in rms])))
    bpd = bytes_per_decision(k_bar, P, A, A)
    dec_per_launch = dec / cx.world / steps / (1 if streams else parts)   # per GPU (concurrent maps: all launches of a step together)
    out = {"workload": desc, "value": dec / (ms / 1000.0), "unit": "decisions/s", "ms_per_step": ms / steps, "timed_region_s": ms / 1000.0,
           "steps": steps, "warmup": warmup, "ticks_per_step": ticks, "n_envs_per_gpu": B, "maps": parts, "q_cap": q_cap, "lanes_per_env": lanes,
           "kernel": variant, "kernel_ms": kern_ms, "decisions_per_launch": dec_per_launch, "train_ticks_per_decision": k_bar,
           "bytes_per_decision": bpd, "ticks": n_ticks,
           "episodes": episodes, "arrived_trains_per_episode": arrived / max(episodes, 1), "trains": T,
           "forced_stop_share": forced / max(dec, 1), "stop_action_share": stops / max(dec, 1),
           "abandoned_episode_share": aborted / max(episodes, 1), "q_rows_max": q_rows_max,
           "l2": (f"L2 flushed between the timed steps (256 MB written, inside the timed region); env state + Q tables {state_mb:.0f} MB per GPU"
                  if flushed else
                  f"inputs larger than L2: {state_mb:.0f} MB of env state + Q tables per GPU vs 126 MB L2, GBs touched per launch"),
           "gpu_launches": steps * parts * (2 if shared else 1),
           "concurrency": (f"{parts} launches per step on {parts} streams, concurrent" if streams else "one launch per step")}
    if shared:
        out["collective"] = {"op": "all_reduce(sum) of int64 step sums + int32 step counts, then sfl_shared_q_apply_to",
                             "backend": "nccl" if cx.world > 1 else "none (1 GPU)", "bytes_per_step": shared_cells * 12,
                             "schedule": "overlapped: runs on a second stream during the next launch, TD steps folded in one step late",
                             "ms_alone": sync_ms, "share_of_step_if_not_overlapped": sync_ms / max(step_ms, 1e-9)}
    return out


def run_e2e(cx: Ctx, wl: str, args, ticks: int, episodes: int) -> dict:
    """End-to-end arm: the call the reference's scripts make -- DistrQLearning.learn(num_episodes, ...) (main.py:63) -- per map,
    wall clock, host<->device copies (hyper-parameter block up; counters, episode logs down) inside the timed region."""
    torch = cx.torch
    from switchfl_b200 import api
    fixture, envs, q_cap, _ = WORKLOADS[wl]
    fxs = workload_fixtures(fixture_path(fixture))
    B = args.envs or envs
    Bp = B // len(fxs)
    B = Bp * len(fxs)
    q_cap = args.q_cap or q_cap
    models = []
    for k, fx in enumerate(fxs):
        env = api.ASyncSwitchEnv(api.RailEnv(fx), max_steps=100_000, n_envs=Bp, device=cx.dev, q_cap=q_cap, ep_cap=max(episodes, 2),
                                 shared_q=(wl == "c5"), _engine_kwargs={"lanes": args.lanes or None, "cta_warps": args.cta_warps or None})
        m = api.DistrQLearning(env=env, seeds=np.arange(Bp, dtype=np.uint64) + np.uint64(SEED + cx.rank * B + k * Bp), dist=cx.dist, **HP)
        m.ticks_per_launch = ticks
        models.append(m)
    def learn_all(n_ep):
        if len(models) > 1:                                               # several maps: concurrently, one stream per learner
            api.learn_concurrently(models, n_ep, None, 0, None)
        else:
            models[0].learn(num_episodes=n_ep, out_dir=None, checkpoint_freq=0)

    learn_all(1)                                                          # warm-up: one short learn() (allocations, first launches)
    for m in models:
        m.env.engine.reset_io_counters()
        m.total_decisions = 0
    cx.barrier()
    w0 = time.perf_counter()
    learn_all(episodes)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - w0
    dec = sum(m.total_decisions for m in models)
    launches = sum(m.env.engine.n_launches for m in models)
    h2d = sum(m.env.engine.h2d_bytes for m in models)
    d2h = sum(m.env.engine.d2h_bytes for m in models)
    for m in models:
        m.env.engine.close()
    del models
    torch.cuda.empty_cache()
    (e2e_s,), (dec,) = cx.reduce([e2e_s], [dec])
    return {"value": dec / e2e_s, "unit": "decisions/s", "h2d_bytes_per_step": h2d // max(launches, 1), "d2h_bytes_per_step": d2h // max(launches, 1),
            "api": (f"DistrQLearning.learn(num_episodes={episodes}, out_dir=None, checkpoint_freq=0)" if len(fxs) == 1 else
                    f"api.learn_concurrently({len(fxs)} learners, num_episodes={episodes}): learn() per map, one thread + stream each"), "wall_s": e2e_s,
            "launches": launches, "step": f"one k_run launch of {ticks} ticks; bytes are the totals copied inside learn() divided by its launches"}


def run_ours(args):
    load_package()
    cx = Ctx()
    wl = args.workload
    ticks = args.ticks or TICKS[wl]
    sampler = ClockSampler(cx.local) if cx.rank == 0 else None
    main = run_block(cx, wl, args, args.steps, args.warmup, sampler=sampler, flush_l2=args.flush_l2)
    clocks = sampler.stop() if sampler else None
    # e2e: about as many flatland ticks per env as the device-resident arm ran
    fx0 = workload_fixtures(fixture_path(WORKLOADS[wl][0]))[0]
    ep = args.e2e_episodes or max(2, int(0.8 * args.steps * ticks / int(fx0["max_episode_steps"])))
    e2e = run_e2e(cx, wl, args, ticks, ep)
    extra = {}
    for name in [x for x in args.extra.split(",") if x and x != wl]:
        extra[name] = run_block(cx, name, args, max(3, args.steps // 2), max(3, args.warmup))
    if cx.rank != 0:
        if cx.dist is not None:
            cx.dist.destroy_process_group()
        return
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = main["decisions_per_launch"] * main["bytes_per_decision"] / (main["kernel_ms"] / 1000.0) / 1e9
    kc = kernel_counters(wl) or {}
    traffic = kc.get("dram_bytes_per_launch") if kc.get("ticks") == ticks and kc.get("envs") == main["n_envs_per_gpu"] else None
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "traffic_source": (kc.get("source", "") + " (committed ncu capture, NOT this run)") if traffic else None,
            "kernel": main["kernel"], "bytes_per_decision": main["bytes_per_decision"], "kernel_ms": main["kernel_ms"], "peak_source": peak_src,
            "note": "byte model of SURVEY 8d; the kernel keeps the env state in shared memory for the launch and is bound by "
                    "instruction issue / dependent-load latency of the serial per-env decision chain, not by HBM (see `issue`)"}
    if kc.get("warp_inst_per_decision"):
        sm_hz = 1e6 * ((clocks or {}).get("sm_mhz") or 1965.0)
        dps_gpu = main["value"] / cx.world
        roof["issue"] = {"warp_inst_per_decision": kc["warp_inst_per_decision"], "threads_per_inst": kc.get("threads_per_inst"),
                         "achieved_warp_inst_per_s": kc["warp_inst_per_decision"] * dps_gpu, "peak_warp_inst_per_s": 148 * 4 * sm_hz,
                         "frac": kc["warp_inst_per_decision"] * dps_gpu / (148 * 4 * sm_hz),
                         "source": kc.get("source", "") + " (committed ncu capture, NOT this run); peak = 148 SMs x 4 schedulers x SM clock"}
    cfg = {k: main[k] for k in ("workload", "n_envs_per_gpu", "maps", "ticks_per_step", "q_cap", "lanes_per_env", "kernel", "decisions_per_launch",
                                "train_ticks_per_decision", "ticks", "episodes", "trains", "arrived_trains_per_episode",
                                "forced_stop_share", "stop_action_share", "abandoned_episode_share", "q_rows_max", "l2", "timed_region_s")}
    cfg["sharding"] = ("envs by seed range, no data-path collective" if wl != "c5" else
                       "envs by seed range; per step one integer all-reduce (sum) of the shared table's accumulators")
    if "collective" in main:
        cfg["collective"] = main["collective"]
    line = {"metric": METRIC, "value": main["value"], "unit": "decisions/s", "n_gpus": cx.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": cfg, "roofline": roof, "e2e": e2e, "gpu_launches": main["gpu_launches"], "clocks": clocks,
            "extra": extra}
    if cx.world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        d, busy, wall, eps = cpu_sample(args.cpu_seconds, cores)
        line["cpu_baseline"] = {"value": d / busy, "unit": "decisions/s", "cores": cores, "kind": "port",
                                "sample": f"{cores} processes x about {args.cpu_seconds:.0f} s of oracle learn() episodes on the same map "
                                          f"({eps} episodes, {d} decisions), one seed per process as hyperparam_tuning.py:85-91",
                                "note": CPU_NOTE}
    print(json.dumps(line))
    if cx.dist is not None:
        cx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS),
                    help="headline workload: c4 = BASELINE.json configs[3] (default), c2 = configs[1], c3 = configs[2], c5 = configs[4]")
    ap.add_argument("--extra", default="c2,c3,c5", help="comma list of further workloads measured in the same run (reported under `extra`)")
    ap.add_argument("--envs", type=int, default=0, help="environments per GPU of the headline workload (0 = the workload's own)")
    ap.add_argument("--ticks", type=int, default=0, help="flatland ticks per env per step of the headline workload (0 = its own: 1024, C2 8192)")
    ap.add_argument("--q-cap", type=int, default=0, help="Q hash rows per environment (0 = the workload's own)")
    ap.add_argument("--lanes", type=int, default=0, help="lanes of a warp per environment (0 = library default for the batch size)")
    ap.add_argument("--cta-warps", type=int, default=0, help="warps per CTA of the hot-path kernel (0 = library default)")
    ap.add_argument("--roomy", type=int, default=-1, help="large-map learn kernel variant: 1 = the 4-CTA/SM build, 0 = the 7-CTA/SM build, -1 = library default")
    ap.add_argument("--flush-l2", default="auto", choices=["auto", "on", "off"],
                    help="write 256 MB between the timed steps (auto: when the whole state is under 1 GiB)")
    ap.add_argument("--e2e-episodes", type=int, default=0, help="episodes per env of the end-to-end learn() call (0 = about as many ticks as the timed steps)")
    ap.add_argument("--cpu-seconds", type=float, default=4.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the headline workload's environments hold after the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path's outputs; the reference arm has none")
    global FIXTURE
    FIXTURE = fixture_path(WORKLOADS[args.workload][0])
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
