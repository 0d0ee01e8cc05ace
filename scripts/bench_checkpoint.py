#!/usr/bin/env python
"""bench_checkpoint.py -- what writing every learner's checkpoints costs learn() on a C3 grid.

    python scripts/bench_checkpoint.py [--envs B] [--old-envs B_OLD] [--episodes E] [--freq F] [--reps R]

One C3 map (``mapgen.c3_fixture(64)``: 80x80, 15 trains, the reference's hyperparam_tuning.py map) with B learners (default
256: one seed's engine of a grid of a few hundred points, each its own learner, bench.py's hyper-parameters, seeds
450565 + i, ``default_q_cap`` rows per table).  ``learn(E, checkpoint_freq=F)`` in four arms, alternated rep by rep:
  none      no checkpoint files (out_dir=None, no env_out_dirs): the learning alone;
  batched   every learner's six checkpoint files into its own directory (``env_out_dirs``): one compaction of all tables on the
            device per checkpoint, copied to pinned staging, written by the writer thread while the next episodes run;
  per_env   the way before it, at the same cadence, on B_OLD learners (default 32, labelled): per environment one
            ``export_q`` (the whole hash image downloaded and scanned on the host, keys decoded row by row) and ``save``;
  none_old  no checkpoint files on B_OLD learners: the baseline of per_env.
Every arm builds its engine before the clock starts; a rep's time is learn()'s wall clock, files written included.
After the reps, on the batched arm's final tables: the compaction kernel's device time (CUDA events around
``sfl_export_q_batch``, median of 20), the bytes and device time of the copy to the host, and the host time to turn one
checkpoint into every learner's files.  Records the card's name and power limit in the same call.  Prints ONE JSON line;
writes the checkpoint files into a temporary directory, nothing into the source tree.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from __graft_entry__ import load_package  # noqa: E402

load_package()
from switchfl_b200 import api, backend, mapgen  # noqa: E402

HP = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)   # bench.py
SEED = 450565
T0 = time.time()


def log(msg):
    print(f"[{time.time() - T0:7.1f} s] {msg}", file=sys.stderr, flush=True)


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return {"name": out[0].strip(), "power_limit_w": float(out[1])}


def per_env_checkpoint(self, writer, targets, cut, cum_reward, arrived, delays, num_malf):
    """The checkpoint as learn() wrote it for the primary environment before the batched export, for every target."""
    eng = self.env.engine
    for i, d in targets:
        q = eng.export_q(i, include_init=self._q_inited, default_q=self._default_q_of(i))
        api._dump_q(q, os.path.join(d, f"checkpoint_{cut + 1}.pkl"))
        np.savez_compressed(os.path.join(d, f"cum_reward_checkpoint_{cut + 1}.npz"), x=cum_reward[i])
        np.savez_compressed(os.path.join(d, f"arrived_trains_checkpoint_{cut + 1}.npz"), x=arrived[i, :cut])
        np.savez_compressed(os.path.join(d, f"delays_checkpoint_{cut + 1}.npz"), x=delays[i, :cut])
        np.savez_compressed(os.path.join(d, f"trains_at_dest_checkpoint_{cut + 1}.npz"), x=[])
        np.savez_compressed(os.path.join(d, f"num_malfunctions_checkpoint_{cut + 1}.npz"), x=num_malf[i, :cut])


def model(rail_env, n):
    env = api.ASyncSwitchEnv(rail_env, max_steps=100_000, n_envs=n, device="cuda:0", ep_cap=16)
    return api.DistrQLearning(env=env, **HP, seed=SEED)


def run_arm(arm, rail_env, args, tmp, rep):
    import torch
    n = args.old_envs if arm in ("per_env", "none_old") else args.envs
    m = model(rail_env, n)
    dirs = None
    if arm in ("batched", "per_env"):
        dirs = [os.path.join(tmp, f"{arm}_{rep}", f"env_{i}") for i in range(n)]
    if arm == "per_env":
        m._checkpoint = types.MethodType(per_env_checkpoint, m)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.learn(args.episodes, None, args.freq, None, env_out_dirs=dirs)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    decisions = int(m.env.engine.counters()["decisions"].sum())
    return m, dt, decisions


def measure_export(m, tmp):
    """Device and host cost of one checkpoint of every learner, on the tables ``m`` ended with."""
    import torch
    eng = m.env.engine
    B, a_max = eng.n_envs, eng.sizes.a_max
    snap = eng.compact_q(0, B, {})                                        # allocates the device buffers
    snap.wait()
    dev = eng._qc
    ptr = lambda name: C.c_void_p(dev[name].data_ptr())
    total = int(snap.off[-1])
    stream = torch.cuda.current_stream()
    kernel_ms = []
    for _ in range(20):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        eng._ck(eng.lib.sfl_export_q_batch(eng.ctx, 0, B, ptr("off"), ptr("keys"), ptr("vals"), C.c_uint64(max(total, 1)),
                                           ptr("found"), eng._stream()))
        b.record(stream)
        b.synchronize()
        kernel_ms.append(a.elapsed_time(b))
    host = {k: torch.empty(v.numel(), dtype=v.dtype, pin_memory=True) for k, v in dev.items() if k != "off"}
    copy_ms = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        host["keys"][:total].copy_(dev["keys"][:total], non_blocking=True)
        host["vals"][:total * a_max].copy_(dev["vals"][:total * a_max], non_blocking=True)
        host["found"][:B].copy_(dev["found"][:B], non_blocking=True)
        b.record(stream)
        b.synchronize()
        copy_ms.append(a.elapsed_time(b))
    nbytes = total * (4 + 8 * a_max) + 4 * B
    t0 = time.perf_counter()
    init = eng.map.q_init_rows(0.0)
    d = os.path.join(tmp, "one_checkpoint")
    for i in range(B):
        os.makedirs(os.path.join(d, f"env_{i}"), exist_ok=True)
        api._dump_q(snap.table(i, init), os.path.join(d, f"env_{i}", "checkpoint.pkl"))
        for name, x in (("cum_reward", m.metrics["cum_reward"][i]), ("arrived_trains", m.metrics["arrived_trains"][i]),
                        ("delays", m.metrics["delays"][i]), ("trains_at_dest", []), ("num_malfunctions", m.metrics["num_malfunctions"][i])):
            np.savez_compressed(os.path.join(d, f"env_{i}", f"{name}_checkpoint.npz"), x=x)
    host_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    n_old = min(B, 16)
    for i in range(n_old):
        eng.export_q(i, include_init=True, default_q=0.0)
    export_q_s = (time.perf_counter() - t0) / n_old
    rows = np.diff(snap.off)
    return {"rows_total": total, "rows_per_env_mean": float(rows.mean()), "rows_per_env_max": int(rows.max()),
            "q_cap": int(eng.cfg.q_cap), "table_bytes_per_env": int(eng.cfg.q_cap) * int(eng.sizes.q_stride) * 8,
            "compact_kernel_ms": kernel_ms, "compact_kernel_ms_median": float(np.median(kernel_ms)),
            "bytes_to_host_per_checkpoint": nbytes, "copy_to_host_ms_median": float(np.median(copy_ms)),
            "host_write_s_per_checkpoint": host_s, "host_write_ms_per_env": 1e3 * host_s / B,
            "export_q_ms_per_env": 1e3 * export_q_s, "export_q_bytes_per_env": int(eng.cfg.q_cap) * int(eng.sizes.q_stride) * 8}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--old-envs", type=int, default=32)
    ap.add_argument("--episodes", type=int, default=30)
    ap.add_argument("--freq", type=int, default=10)
    ap.add_argument("--reps", type=int, default=1)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_checkpoint.py measures the CUDA path: no CUDA device")
    info = card()
    rail_env = api.RailEnv(mapgen.c3_fixture(64))
    arms = ("none", "batched", "none_old", "per_env")
    res = {a: {"wall_s": [], "decisions": []} for a in arms}
    last = None
    with tempfile.TemporaryDirectory() as tmp:
        log("warm-up")
        run_arm("none", rail_env, argparse.Namespace(**{**vars(args), "episodes": 2}), tmp, -1)
        for rep in range(args.reps):
            for arm in arms:
                m, dt, dec = run_arm(arm, rail_env, args, tmp, rep)
                res[arm]["wall_s"].append(dt)
                res[arm]["decisions"].append(dec)
                log(f"rep {rep} {arm}: {dt:.2f} s, {dec} decisions")
                if arm == "batched":
                    last = m
                else:
                    m.env.engine.close()
        log("export costs")
        exp = measure_export(last, tmp)
    checkpoints = len([t for t in range(args.episodes) if (t + 1) % args.freq == 0])
    for arm in arms:
        r = res[arm]
        r["envs"] = args.old_envs if arm in ("per_env", "none_old") else args.envs
        r["wall_s_median"] = float(np.median(r["wall_s"]))
    for arm, base in (("batched", "none"), ("per_env", "none_old")):
        res[arm]["overhead_s_per_checkpoint"] = (res[arm]["wall_s_median"] - res[base]["wall_s_median"]) / max(checkpoints, 1)
    out = {"card": info, "map": "c3_rail80_s64 (mapgen.c3_fixture(64))", "episodes": args.episodes, "checkpoint_freq": args.freq,
           "checkpoints": checkpoints, "reps": args.reps, "arms": res, "export": exp,
           "note": f"per_env and none_old run {args.old_envs} learners (reduced), none and batched {args.envs}; each pair learns the "
                   "same episodes, so its difference is what the checkpoints cost learn()"}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
