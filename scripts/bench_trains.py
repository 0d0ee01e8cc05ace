#!/usr/bin/env python
"""bench_trains.py -- switch-agent decisions/sec on a map with more than 64 trains (the two-word train-set kernels).

    python scripts/bench_trains.py [--gpus 1] [--steps K] [--warmup W]

Workload: ``rail100_t100`` (``mapgen.t100_fixture``: the C4 rail network with 100 trains, the size of the reference's
100-train evaluation), 3552 lockstep environments -- one 32-lane group each -- each an independent distributed-Q learner
with bench.py's hyper-parameters, learn mode.  3552 = 148 SMs x 24: an SM holds 12 two-warp CTAs of the 80-register kernel
(shared memory, 8.1 KB per environment, would allow 13), so the batch is exactly one wave.  A batch a little above a wave
leaves the remainder to run alone for a whole launch: on B200, 4096 environments gave 1.93e8 decisions/s where one full
wave (3848, with the 72-register build of this kernel) gave 2.99e8.  A step is one k_run launch of ``--ticks`` flatland ticks
per environment, timed with CUDA events on resident state, after ``--warmup`` untimed launches (bench.py's conventions).

Prints ONE JSON line: the device-timed decisions/s and, from the same call, the card and its power limit, the kernel
instantiation, its registers (cuobjdump -res-usage of the built library) and the environments resident per SM that
follow from them, arrivals per episode, the forced-STOP share, the per-phase split of the instrumented kernel
(sfl_set_phase_clock: phase 0 is the whole train tick, the motion check included) and ``DistrQLearning.learn()`` end to
end on the same map.  Writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from __graft_entry__ import LIB, load_package  # noqa: E402

METRIC = "switch_agent_decisions_per_sec"
HP = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)   # bench.py
SEED = 450565
ENVS = 3552                      # one full wave on a 148-SM B200 (see above)
Q_CAP = 131072                   # Q hash rows per environment: q_rows_max in the output says how many a run used
TICKS = 1024
PHASES = ("tick", "observe", "act", "apply", "update", "reset")


def card():
    """Name and power limit of GPU 0 (nvidia-smi), read in the same call as the measurement."""
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return {"name": out[0].strip(), "power_limit_w": float(out[1]), "sm_max_mhz": float(out[2])}


def kernel_registers(template: str) -> int:
    """Registers of the k_run instantiation named by sfl_describe_launch, from the library's own cubin."""
    m = dict(kv.split("=") for kv in re.search(r"<(.*)>", template).group(1).split(","))
    kind = {"learn": 0, "greedy": 1, "full": 2}[m["KIND"]]
    b = lambda k: "1" if m.get(k, "0") == "1" else "0"
    sym = f"_Z5k_runILi{m['G']}ELi{kind}ELb{b('TH')}ELb{b('SQ')}ELb{b('ONE')}ELb{b('ROOMY')}ELi{m.get('NW', '1')}EEvN3sfl5KArgsE"
    cuobjdump = os.path.join(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")), "cuobjdump")
    out = subprocess.run([cuobjdump, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    hit = re.search(re.escape(sym) + r":\s*\n\s*REG:(\d+)", out)
    if not hit:
        raise SystemExit(f"bench_trains.py: {sym} not found in {LIB}")
    return int(hit.group(1))


def resident_envs_per_sm(regs: int, threads: int, smem: int, lanes: int) -> dict:
    """CTAs (and environments) one SM holds: sm_100 limits -- 64K registers allocated per warp in units of 256, 2048 threads,
    32 CTAs, 228 KB of shared memory with 1 KB reserved per CTA."""
    warps = threads // 32
    by_regs = 65536 // (warps * ((regs * 32 + 255) // 256 * 256))
    by_threads = 2048 // threads
    by_smem = (228 * 1024) // (smem + 1024)
    ctas = min(by_regs, by_threads, by_smem, 32)
    return {"ctas": ctas, "envs": ctas * threads // lanes, "limited_by": min((by_regs, "registers"), (by_threads, "threads"),
                                                                             (by_smem, "shared memory"), (32, "CTA slots"))[1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--ticks", type=int, default=TICKS)
    ap.add_argument("--envs", type=int, default=ENVS)
    ap.add_argument("--phase-steps", type=int, default=4, help="launches of the instrumented kernel for the per-phase split")
    args = ap.parse_args()
    if args.gpus != 1:
        raise SystemExit("bench_trains.py measures one GPU")
    load_package()
    import torch
    from switchfl_b200 import api, backend, mapgen
    if not torch.cuda.is_available():
        raise SystemExit("bench_trains.py: no CUDA device; the hot path has no CPU fallback")
    dev = "cuda:0"
    fx = mapgen.t100_fixture()
    rm = backend.RailMap(fx, device_bfs=0)
    gpu = card()
    B = args.envs

    def engine(**kw):
        eng = backend.Engine(rm, n_envs=B, device=dev, q_cap=Q_CAP, ep_cap=4, **kw)
        eng.set_hparams(**HP, seeds=np.arange(B, dtype=np.uint64) + np.uint64(SEED), episodes=-1)
        eng.reset()
        eng.enable_q_init(True)
        return eng

    def totals(eng):
        c = eng.counters()
        return np.array([int(c[k].sum()) for k in ("decisions", "ticks", "episodes", "forced_stops", "arrived_trains", "aborted")], np.int64)

    # ---- device-resident arm: k_run learn launches, CUDA events
    eng = engine()
    launch = eng.describe_launch(backend.MODE_LEARN)
    for _ in range(args.warmup):
        eng.run(backend.MODE_LEARN, args.ticks)
    torch.cuda.synchronize()
    t0 = totals(eng)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(args.steps):
        eng.run(backend.MODE_LEARN, args.ticks)
    stop.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(stop)
    dec, ticks, episodes, forced, arrived, aborted = totals(eng) - t0
    eng.check_errors()
    q_rows_max = int(eng.counters()["q_rows"].max())
    eng.close()
    del eng
    torch.cuda.empty_cache()

    kernel = launch.split(" ")[0]
    lp = dict(kv.split("=") for kv in launch.split(" ")[1:])
    regs = kernel_registers(kernel)
    occ = resident_envs_per_sm(regs, int(lp["block"]), int(lp["smem"]), int(re.search(r"G=(\d+)", kernel).group(1)))

    # ---- per-phase split: the instrumented (full) kernel on the same batch
    eng = engine(phase_clock=True)
    for _ in range(args.phase_steps):
        eng.run(backend.MODE_LEARN, args.ticks)
    eng.check_errors()
    ph = eng.counters()["phase_cycles"].astype(np.float64).sum(axis=0)
    phase_kernel = eng.kernel_variant(backend.MODE_LEARN)
    eng.close()
    del eng
    torch.cuda.empty_cache()

    # ---- end to end: DistrQLearning.learn() on the same map and batch
    ep = max(2, int(0.8 * args.steps * args.ticks / int(fx["max_episode_steps"])))
    env = api.ASyncSwitchEnv(api.RailEnv(fx), max_steps=100_000, n_envs=B, device=dev, q_cap=Q_CAP, ep_cap=ep)
    m = api.DistrQLearning(env=env, seeds=np.arange(B, dtype=np.uint64) + np.uint64(SEED), **HP)
    m.ticks_per_launch = args.ticks
    m.learn(num_episodes=1, out_dir=None, checkpoint_freq=0)                # warm-up
    m.total_decisions = 0
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    m.learn(num_episodes=ep, out_dir=None, checkpoint_freq=0)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - w0
    e2e_dec = m.total_decisions
    env.engine.close()

    line = {"metric": METRIC, "value": dec / (ms / 1000.0), "unit": "decisions/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "dtype": "f64", "data": "synthetic",
            "gpu": gpu,
            "config": {"workload": f"{fx['name']}: 100x100 C4 rail network, {rm.trains.T} trains, {rm.tab.S} switches, {rm.tab.NP} ports, "
                                   "malfunctions 0.01 / 5-15, distributed Q-learning, learn mode",
                       "n_envs": B, "ticks_per_step": args.ticks, "q_cap": Q_CAP, "q_rows_max": q_rows_max},
            "kernel": kernel, "launch": launch, "registers": regs, "resident_per_sm": occ,
            "decisions": int(dec), "ticks": int(ticks), "episodes": int(episodes),
            "arrived_trains_per_episode": arrived / max(episodes, 1), "forced_stop_share": forced / max(dec, 1),
            "abandoned_episode_share": aborted / max(episodes, 1),
            "phase_split": {"kernel": phase_kernel, "launches": args.phase_steps,
                            "share": {n: float(x) for n, x in zip(PHASES, ph / max(ph.sum(), 1.0))},
                            "note": "SM cycles per phase of the instrumented kernel; 'tick' is the whole per-tick train phase "
                                    "(plan pop, motion check, state machine, semaphore bookkeeping)"},
            "e2e": {"value": e2e_dec / e2e_s, "unit": "decisions/s", "api": f"DistrQLearning.learn(num_episodes={ep}, out_dir=None, checkpoint_freq=0)",
                    "wall_s": e2e_s, "decisions": int(e2e_dec)}}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
