#!/usr/bin/env python
"""Dynamics of a map fixture under the free-running learner: arrivals per episode, forced-STOP share, abandoned episodes.

Development tooling (CPU): drives the host build of the device sources (tests/emul, test infrastructure) so that map
generator parameters can be tuned on the GPU-less box.  The numbers to compare against are the reference's learning
curves (BASELINE.md: about 5.8 of 15 trains arrive at episode 0 with epsilon 0.5, about 14.7 of 15 once trained).

    python tools/map_stats.py tests/golden/c4_synth100_t50.fixture.npz [--envs 8] [--episodes 3]
    python tools/map_stats.py mapgen.t100_fixture                # a map generated from its seed by a mapgen function
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402

load_package()
from switchfl_b200 import backend, mapgen  # noqa: E402

HP = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)


def stats(fx: dict, n_envs: int = 8, n_ep: int = 3, seed0: int = 450565, q_cap: int = 65536, hp: dict = HP, dec_cap: int = 200000) -> dict:
    from tests.emulated import EmulEngine
    rm = backend.RailMap(fx)
    T = rm.trains.T
    eng = EmulEngine(rm, n_envs=n_envs, q_cap=q_cap, dec_cap=dec_cap, ep_cap=n_ep + 1)
    eng.set_hparams(**hp, seeds=np.arange(n_envs) + seed0, episodes=n_ep)
    eng.reset()
    eng.enable_q_init(True)
    eng.run(backend.MODE_LEARN, 10_000_000)
    c = eng.counters()
    _, log, _ = eng.episode_log()
    forced = chosen = total = 0
    for i in range(n_envs):
        dec, _, _ = eng.trace(i)
        A = rm.tab.sw_A[dec["sw"]]
        stop_bit = 1 << (A - 1)
        forced += int((dec["mask"] == stop_bit).sum())
        chosen += int((dec["action"] == A - 1).sum())
        total += len(dec)
    out = {
        "name": fx["name"], "S": rm.tab.S, "NP": rm.tab.NP, "T": T, "max_episode_steps": int(fx["max_episode_steps"]),
        "arrived_per_episode": [float(log["arrived"][:, e].mean()) for e in range(n_ep)],
        "arrived_frac_ep0": float(log["arrived"][:, 0].mean()) / T,
        "decisions_per_episode": float(log["decisions"][:, :n_ep].mean()),
        "ticks_per_episode": float(log["ticks"][:, :n_ep].mean()),
        "forced_stop_share": forced / max(total, 1), "stop_chosen_share": chosen / max(total, 1),
        "aborted_share": float(c["aborted"].sum()) / (n_envs * n_ep),
        "train_ticks_per_decision": float(c["train_ticks"].sum()) / max(int(c["decisions"].sum()), 1),
        "q_rows_max": int(c["q_rows"].max()), "err_bits": int(np.bitwise_or.reduce(c["err"])),
    }
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("fixture", nargs="+", help="fixture .npz, or mapgen.<function> for a generated map")
    ap.add_argument("--envs", type=int, default=8)
    ap.add_argument("--episodes", type=int, default=3)
    args = ap.parse_args()
    for path in args.fixture:
        fx = getattr(mapgen, path[len("mapgen."):])() if path.startswith("mapgen.") else mapgen.load_fixture(path)
        s = stats(fx, args.envs, args.episodes)
        print({k: (round(v, 3) if isinstance(v, float) else v) for k, v in s.items()})


if __name__ == "__main__":
    main()
