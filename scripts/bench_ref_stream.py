#!/usr/bin/env python
"""bench_ref_stream.py -- what learning on the reference's random stream costs: Philox learn kernel vs the full kernel on
numpy's PCG64 stream (``Engine(rng="reference")``).

    python scripts/bench_ref_stream.py [--steps K] [--warmup W] [--ticks N]

Two workloads, bench.py's hyper-parameters, learn mode: C4 (``mapgen.c4_fixture``) at the benchmark batch of 8192
environments, and ``rail100_t100`` (``mapgen.t100_fixture``) at 3552 (one wave, see bench_trains.py).  Per workload both arms
are built side by side and timed alternately: a step is one k_run launch of ``--ticks`` flatland ticks per environment on
resident state, timed with CUDA events after ``--warmup`` untimed launches; the arms take turns step by step.

Also reported, from the same call: the share of decisions that explored (counted exactly on a 32-environment sample:
the host replays numpy's generator over the sample's decision trace and checks that it lands on the device's final
stream state), the kernel instantiations, and the card with its power limit.  Prints ONE JSON line; writes nothing into
the source tree.
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
WORKLOADS = (("c4", 8192, 16384), ("t100", 3552, 131072))       # (map, environments, Q rows per environment)


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


def make(backend, rm, n, q_cap, rng):
    eng = backend.Engine(rm, n_envs=n, q_cap=q_cap, ep_cap=4, rng=rng)
    eng.set_hparams(**HP, seeds=np.arange(n) + SEED, episodes=-1)
    eng.reset()
    eng.enable_q_init(True)
    return eng


def explored_share(backend, rm, ticks):
    """Exact share of exploring decisions on 32 environments, self-checked against the device's stream state."""
    n = 32
    eng = backend.Engine(rm, n_envs=n, q_cap=16384 if rm.trains.T <= 64 else 131072, ep_cap=4, dec_cap=ticks * rm.trains.T, rng="reference")
    eng.set_hparams(**HP, seeds=np.arange(n) + SEED, episodes=1)
    eng.reset()
    eng.enable_q_init(True)
    eng.run(backend.MODE_LEARN, ticks)
    eng.check_errors()
    logged = eng.counters()["n_dec_logged"]
    assert (logged <= eng.cfg.dec_cap).all(), "trace buffer too small"
    trace = eng.buf["trace_dec"][:n * eng.cfg.dec_cap * backend.DEC_DT.itemsize].cpu().numpy().view(backend.DEC_DT).reshape(n, -1)
    dec_total = explored = 0
    for i in range(n):
        dec = trace[i, :int(logged[i])]
        r = np.random.default_rng(SEED + i)
        count = np.zeros(rm.tab.S, np.int64)
        for s in dec["sw"]:
            u = r.random()
            if u < HP["epsilon"] * HP["epsilon_decay_rate"] ** int(count[s]):
                r.integers(0, 2 ** 31 - 1)
                explored += 1
            count[s] += 1
        assert eng.rng_state(i) == r.bit_generator.state, f"env {i}: the host replay of the stream diverged"
        dec_total += len(dec)
    eng.close()
    return explored / max(dec_total, 1), dec_total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ticks", type=int, default=1024)
    args = ap.parse_args()
    load_package()
    import torch
    from switchfl_b200 import backend
    if not torch.cuda.is_available():
        raise SystemExit("bench_ref_stream.py needs a CUDA device")
    result = {"card": card(), "steps": args.steps, "warmup": args.warmup, "ticks": args.ticks, "workloads": {}}
    for name, n, q_cap in WORKLOADS:
        rm = backend.RailMap(fixture(name), device_bfs=0)
        arms = {rng: make(backend, rm, n, q_cap, rng) for rng in ("philox", "reference")}
        log(f"{name}: {n} environments, both arms built")
        for eng in arms.values():
            for _ in range(args.warmup):
                eng.run(backend.MODE_LEARN, args.ticks)
        torch.cuda.synchronize()
        ms = {k: 0.0 for k in arms}
        dec = {k: 0 for k in arms}
        for _ in range(args.steps):
            for rng, eng in arms.items():                                 # alternate the arms step by step
                d0, _ = eng.total_decisions()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                eng.run(backend.MODE_LEARN, args.ticks)
                b.record()
                b.synchronize()
                ms[rng] += a.elapsed_time(b)
                d1, _ = eng.total_decisions()
                dec[rng] += d1 - d0
                log(f"{name} {rng}: {d1 - d0} decisions in {a.elapsed_time(b):.1f} ms")
        out = {}
        for rng, eng in arms.items():
            eng.check_errors()
            out[rng] = {"kernel": eng.describe_launch(backend.MODE_LEARN), "decisions": int(dec[rng]),
                        "decisions_per_sec": dec[rng] / (ms[rng] / 1e3)}
            eng.close()
        out["reference_over_philox"] = out["reference"]["decisions_per_sec"] / out["philox"]["decisions_per_sec"]
        share, sample = explored_share(backend, rm, args.ticks)
        log(f"{name}: explored share {share:.4f} over {sample} decisions")
        out["explored_share"] = share
        out["explored_sample_decisions"] = sample
        out["environments"] = n
        result["workloads"][name] = out
    print(json.dumps(result))


if __name__ == "__main__":
    main()
