#!/usr/bin/env python
"""bench_eval.py -- greedy evaluation of one learned table on many environments: the evaluation kernel (one read-only table
shared by every environment, ``Engine(eval_q=True)``) against the per-environment greedy kernel (a private copy each, what
``load()`` + ``test()`` builds).

    python scripts/bench_eval.py [--reps R] [--learn-episodes E]

For C4 (``mapgen.c4_fixture``) and ``rail100_t100`` (``mapgen.t100_fixture``): a table from a short ``learn()`` (64
environments, ``--learn-episodes`` episodes, bench.py's hyper-parameters; environment 0's table with the optimistic rows),
then one greedy episode per environment, seeds 450565 + i, in these arms, alternated rep by rep in the same call:
  eval_<N>     the evaluation kernel at N environments (BATCHES);
  eval_same    the evaluation kernel at the private arm's batch;
  private      the per-environment greedy kernel at the largest batch whose private tables (``default_q_cap`` rows each, as
               ``load()`` sizes them) fit in 70 % of the free device memory, at most 8192; the table is imported once and
               copied to every environment on the device.
A rep is one launch that runs every environment's episode to its end, timed with CUDA events; the reset before it is not
timed.  The working sets of the private arm exceed the 126 MB L2; the evaluation table fits it.  eval_same and private must
give identical episodes (checked).  Also reported: bytes per environment (env_stride) of both layouts and the time to
build and upload the evaluation table.  Records the card's name and power limit in the same call.  Prints ONE JSON line;
writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import functools
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

load_package()
from switchfl_b200 import api, backend, mapgen  # noqa: E402

HP = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)   # bench.py
SEED = 450565
BATCHES = {"c4": (8192, 32768), "t100": (3552, 8192, 32768)}
PRIVATE_MAX = 8192

T0 = time.time()


def log(msg):
    print(f"[{time.time() - T0:7.1f} s] {msg}", file=sys.stderr, flush=True)


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return {"name": out[0].strip(), "power_limit_w": float(out[1])}


@functools.lru_cache(maxsize=None)
def rail_map(name, device_bfs=None):
    return backend.RailMap(mapgen.c4_fixture() if name == "c4" else mapgen.t100_fixture(), device_bfs=device_bfs)


def learned_table(name, episodes):
    env = api.ASyncSwitchEnv(api.RailEnv(rail_map(name, 0).fixture), max_steps=100_000, n_envs=64)
    m = api.DistrQLearning(env, **HP, seed=SEED)
    m.learn(episodes, None, 0)
    q = dict(m.q_table)
    env.engine.close()
    return q


class Arm:
    def __init__(self, torch, rm, q, n, eval_q):
        self.torch, self.n, self.steps = torch, n, int(rm.fixture["max_episode_steps"]) + 8
        seeds = np.arange(n) + SEED
        if eval_q:
            cap = 1024
            while cap < 2 * len(q) + 2:
                cap *= 2
            self.eng = backend.Engine(rm, n_envs=n, q_cap=cap, ep_cap=1, eval_q=True)
            self.eng.set_hparams(**HP, seeds=seeds, episodes=1)
            self.eng.reset()
            torch.cuda.synchronize()
            t = time.perf_counter()
            self.eng.set_eval_table(q)
            self.table_ms = (time.perf_counter() - t) * 1e3
        else:                                                    # load(): the table into every private table
            self.eng = backend.Engine(rm, n_envs=n, q_cap=api.default_q_cap(rm), ep_cap=1)
            self.eng.set_hparams(**HP, seeds=seeds, episodes=-1)
            self.eng.reset()
            self.eng.import_q(0, q)
            blocks = self.eng.buf["state"][:n * self.eng.sizes.env_stride].view(n, -1)
            blocks[1:] = blocks[0]
            self.eng.set_hparams(**HP, seeds=seeds, episodes=1)
        self.keep = not eval_q
        self.ms, self.dec = [], 0

    def rep(self):
        torch, eng = self.torch, self.eng
        eng.reset(keep_q=self.keep, keep_interactions=self.keep)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.run(backend.MODE_GREEDY, self.steps)
        b.record()
        b.synchronize()
        c = eng.counters()
        eng.check_errors()
        assert (c["halted"] == 1).all(), "an episode did not end within one launch"
        self.ms.append(a.elapsed_time(b))
        self.dec = int(c["decisions"].sum())

    def result(self):
        _, lg, _ = self.eng.episode_log()
        ms = float(np.median(self.ms))
        return {"environments": self.n, "kernel": self.eng.describe_launch(backend.MODE_GREEDY), "env_stride": int(self.eng.sizes.env_stride),
                "ms": self.ms, "ms_median": ms, "episodes_per_sec": self.n / (ms / 1e3), "decisions_per_sec": self.dec / (ms / 1e3),
                "decisions_per_episode": self.dec / self.n, "mean_arrived": float(lg["arrived"][:, 0].mean())}


def bench_map(torch, name, reps, learn_episodes):
    rm = rail_map(name, 0)
    q = learned_table(name, learn_episodes)
    log(f"{name}: table of {len(q)} rows from a {learn_episodes}-episode learn()")
    probe = backend.Engine(rm, n_envs=1, q_cap=api.default_q_cap(rm), ep_cap=1, bind=False)
    stride = int(probe.sizes.env_stride)
    probe.close()
    free, _ = torch.cuda.mem_get_info()
    n_priv = min(PRIVATE_MAX, int(0.7 * free) // stride // 64 * 64)
    arms = {f"eval_{n}": Arm(torch, rm, q, n, True) for n in BATCHES[name]}
    arms["eval_same"] = Arm(torch, rm, q, n_priv, True)
    arms["private"] = Arm(torch, rm, q, n_priv, False)
    log(f"{name}: arms built, private batch {n_priv} ({stride} bytes per environment)")
    for arm in arms.values():                                    # warm-up: modules, first touch
        arm.rep()
    for arm in arms.values():
        arm.ms = []
    for r in range(reps):
        for k, arm in arms.items():
            arm.rep()
        log(f"{name} rep {r}: " + ", ".join(f"{k} {a.ms[-1]:.1f} ms" for k, a in arms.items()))
    _, le, de = arms["eval_same"].eng.episode_log()
    _, lp, dp = arms["private"].eng.episode_log()
    same = bool(all(np.array_equal(le[f], lp[f]) for f in ("cum_reward", "decisions", "ticks", "arrived", "arrived_mask",
                                                            "arrived_mask_hi", "num_malfunctions")) and np.array_equal(de, dp))
    out = {"trains": rm.trains.T, "table_rows": len(q), "eval_table_bytes": int(arms["eval_same"].eng.sizes.eval_q_bytes),
           "set_eval_table_ms": arms[f"eval_{BATCHES[name][0]}"].table_ms, "private_q_cap": api.default_q_cap(rm),
           "eval_same_equals_private": same, "arms": {k: a.result() for k, a in arms.items()}}
    out["eval_same_over_private"] = out["arms"]["eval_same"]["episodes_per_sec"] / out["arms"]["private"]["episodes_per_sec"]
    for a in arms.values():
        a.eng.close()
        a.eng.buf = {}
    del arms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--learn-episodes", type=int, default=8)
    ap.add_argument("--maps", default="c4,t100")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval.py needs a CUDA device")
    result = {"card": card(), "reps": args.reps, "learn_episodes": args.learn_episodes}
    for name in args.maps.split(","):
        result[name] = bench_map(torch, name, args.reps, args.learn_episodes)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
