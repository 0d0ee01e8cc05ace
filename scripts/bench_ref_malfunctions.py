#!/usr/bin/env python
"""bench_ref_malfunctions.py -- what flatland's malfunction stream costs (``Engine(malfunction_rng="reference")``).

    python scripts/bench_ref_malfunctions.py [--steps K] [--warmup W] [--ticks N] [--reps R]

(a) Schedule generation (``sfl_malf_schedule``: one warp per environment, numpy's MT19937 on the device) on C4
    (``mapgen.c4_fixture``) with 8192 environments and on ``rail100_t100`` (``mapgen.t100_fixture``) with 3552: the call
    is repeated ``--reps`` times after one untimed call, each timed with CUDA events around it (it ends in a synchronise).
(b) Learn decisions/s on C4 with 8192 environments and bench.py's hyper-parameters, three arms built side by side and
    timed alternately, step by step: the reference's epsilon-greedy stream with flatland's malfunctions
    (``rng="reference", malfunction_rng="reference"``), the same stream with Philox malfunctions, and the Philox learn
    kernel.  A step is one k_run launch of ``--ticks`` flatland ticks per environment on resident state, timed with CUDA
    events after ``--warmup`` untimed launches.

Records the card's name and power limit in the same call.  Prints ONE JSON line; writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from __graft_entry__ import load_package  # noqa: E402

HP = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)   # bench.py
SEED = 450565
# (map, environments, Q rows per environment): C4 with bench.py's 65536 rows -- learning runs on without resets here, and
# with 16384 rows every arm, Philox included, ran 40-150x slower from the fourth timed launch on (one B200)
GENERATION = (("c4", 8192, 65536), ("t100", 3552, 131072))
ARMS = {"reference_with_flatland_malfunctions": dict(rng="reference", malfunction_rng="reference"),
        "reference_with_philox_malfunctions": dict(rng="reference"),
        "philox": dict()}

T0 = time.time()


def log(msg):
    print(f"[{time.time() - T0:7.1f} s] {msg}", file=sys.stderr, flush=True)


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return {"name": out[0].strip(), "power_limit_w": float(out[1])}


def fixture(name):
    from switchfl_b200 import mapgen
    return mapgen.c4_fixture() if name == "c4" else mapgen.t100_fixture()


def make(backend, rm, n, q_cap, **kw):
    eng = backend.Engine(rm, n_envs=n, q_cap=q_cap, ep_cap=4, **kw)
    eng.set_hparams(**HP, seeds=np.arange(n) + SEED, episodes=-1)
    eng.reset()
    eng.enable_q_init(True)
    return eng


def generation(torch, backend, name, n, q_cap, reps):
    rm = backend.RailMap(fixture(name), device_bfs=0)
    eng = make(backend, rm, n, q_cap, rng="reference", malfunction_rng="reference")
    times = []
    for rep in range(reps + 1):
        eng._malf_key = None                          # force a regeneration
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng._malf_generate()
        b.record()
        b.synchronize()
        if rep:
            times.append(a.elapsed_time(b))
    lens = [len(eng.malfunction_schedule(i)) for i in range(0, n, max(1, n // 64))]
    out = {"environments": n, "trains": rm.trains.T, "max_episode_steps": int(rm.fixture["max_episode_steps"]),
           "draws_per_env": rm.trains.T * int(rm.fixture["max_episode_steps"]), "ev_cap": int(eng.cfg.ev_cap),
           "max_events": int(eng.max_malfunction_events), "mean_events_sampled": float(np.mean(lens)),
           "ms": times, "ms_median": float(np.median(times))}
    log(f"{name}: schedule generation {out['ms_median']:.3f} ms (median of {reps})")
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ticks", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    load_package()
    import torch
    from switchfl_b200 import backend
    if not torch.cuda.is_available():
        raise SystemExit("bench_ref_malfunctions.py needs a CUDA device")
    result = {"card": card(), "steps": args.steps, "warmup": args.warmup, "ticks": args.ticks, "reps": args.reps,
              "generation": {}, "learn_c4": {}}
    for name, n, q_cap in GENERATION:
        result["generation"][name] = generation(torch, backend, name, n, q_cap, args.reps)
    name, n, q_cap = GENERATION[0]
    rm = backend.RailMap(fixture(name), device_bfs=0)
    arms = {k: make(backend, rm, n, q_cap, **kw) for k, kw in ARMS.items()}
    log(f"{name}: {n} environments, three arms built")
    for eng in arms.values():
        for _ in range(args.warmup):
            eng.run(backend.MODE_LEARN, args.ticks)
    torch.cuda.synchronize()
    ms = {k: 0.0 for k in arms}
    dec = {k: 0 for k in arms}
    for _ in range(args.steps):
        for k, eng in arms.items():                                   # alternate the arms step by step
            d0, _ = eng.total_decisions()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.run(backend.MODE_LEARN, args.ticks)
            b.record()
            b.synchronize()
            ms[k] += a.elapsed_time(b)
            d1, _ = eng.total_decisions()
            dec[k] += d1 - d0
            log(f"{name} {k}: {d1 - d0} decisions in {a.elapsed_time(b):.1f} ms")
    out = {}
    for k, eng in arms.items():
        eng.check_errors()
        c = eng.counters()
        out[k] = {"kernel": eng.describe_launch(backend.MODE_LEARN), "decisions": int(dec[k]),
                  "decisions_per_sec": dec[k] / (ms[k] / 1e3), "episodes": int(c["episodes"].sum())}
        eng.close()
    base = out["philox"]["decisions_per_sec"]
    for k in ARMS:
        out[k]["over_philox"] = out[k]["decisions_per_sec"] / base
    out["environments"] = n
    result["learn_c4"] = out
    print(json.dumps(result))


if __name__ == "__main__":
    main()
