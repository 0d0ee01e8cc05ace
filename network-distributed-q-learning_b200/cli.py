"""The reference's driver scripts on the batched backend (SURVEY.md section 8f row N4).

    python -m switchfl_b200.cli -c config.ini                 # main.py:83-88, same INI schema
    launch_grid(hyperparams, random_seeds, out_dir, ...)      # hyperparam_tuning.py:42-91 without the process fan-out
    launch_eval(exp_dir_list)                                 # eval.py:31-97
    python -m switchfl_b200.cli --eval EXP_DIR... [--num-evals N]

``config.ini`` keeps the reference's sections and keys (hyperparam_tuning.py:51-78): MISC{random_seed, out_dir,
checkpoint_freq, exploit_freq}, ENV{width, height, max_num_cities, max_rails_between_cities, max_rail_pairs_in_city,
number_of_agents, malfunction_rate, min_duration, max_duration}, MODEL{gamma, epsilon, epsilon_decay_rate, lr,
lr_decay_rate, default_q, num_episodes}.  Five optional keys are new: ENV.fixture (a map fixture .npz recorded from
flatland, see tools/record_flatland_fixture.py), MISC.n_envs (lockstep replicas with seeds random_seed + i),
MISC.q_cap (Q hash rows per environment; default: sized from the map, see ``default_q_cap``), MISC.rng (``philox``,
the default, or ``reference``: the reference's own numpy epsilon-greedy stream, see ``ASyncSwitchEnv``) and
MISC.malfunction_rng (``philox``, the default, or ``reference``: flatland's own malfunction stream of the seed).
Without ENV.fixture the map comes from the synthetic generator with the same size / train count / seed, because
flatland's sparse_rail_generator cannot run here (mapgen.py).
"""
from __future__ import annotations

import argparse
import configparser
import os
import time
from itertools import product
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import mapgen, sharding
from .api import ASyncSwitchEnv, DistrQLearning, MalfunctionParameters, ParamMalfunctionGen, RailEnv, learn_concurrently, read_q_table


def fixture_from_env_section(env: Dict[str, str], seed: int) -> dict:
    if env.get("fixture"):
        return mapgen.load_fixture(env["fixture"])
    n = int(env["width"])
    if int(env["height"]) != n:
        raise ValueError("the reference only works on square grids (utils/rail_graph.py:43-48)")
    cities = int(env.get("max_num_cities", 2))
    rails = int(env.get("max_rails_between_cities", 1))
    if rails >= 2:            # double track between the cities (hyperparam_tuning.py:20): the right-hand-running generator
        lines = max(2, min(cities // 3, n // 8))
        return mapgen.rail_fixture(n, int(env["number_of_agents"]), seed, n_rings=2, n_lines=lines, cross_every=10, num_cities=cities)
    chords = max(2, cities * rails * int(env.get("max_rail_pairs_in_city", 1)) // 2)
    return mapgen.make_fixture(n=n, n_trains=int(env["number_of_agents"]), n_chords=chords, seed=seed, num_cities=cities)


def default_device() -> str:
    """``cuda:<LOCAL_RANK>`` (one process per GPU under torchrun), made current for torch."""
    import torch
    local = sharding.world()[2]
    if torch.cuda.is_available():
        torch.cuda.set_device(local)
    return f"cuda:{local}"


def launch_experiment(config_path: str, device: Optional[str] = None, q_cap: Optional[int] = None, env_cls=ASyncSwitchEnv,
                      _engine_kwargs=None, rng: Optional[str] = None, malfunction_rng: Optional[str] = None) -> DistrQLearning:
    """main.py:13-78."""
    start_time = time.time()
    device = device or default_device()
    config = configparser.ConfigParser()
    config.read(config_path)
    misc, envs, mdl = config["MISC"], config["ENV"], config["MODEL"]
    out_dir = misc["out_dir"]
    seed = int(misc["random_seed"])
    mf = ParamMalfunctionGen(MalfunctionParameters(malfunction_rate=float(envs["malfunction_rate"]),
                                                   min_duration=int(envs["min_duration"]), max_duration=int(envs["max_duration"])))
    rail_env = RailEnv(fixture_from_env_section(dict(envs), seed), malfunction_generator=mf)
    if q_cap is None and misc.get("q_cap"):
        q_cap = int(misc["q_cap"])
    rng = rng or misc.get("rng", "philox")
    malfunction_rng = malfunction_rng or misc.get("malfunction_rng", "philox")
    env = env_cls(rail_env, render_mode=None, max_steps=100_000, n_envs=int(misc.get("n_envs", 1)), device=device, q_cap=q_cap,
                  rng=rng, malfunction_rng=malfunction_rng, _engine_kwargs=_engine_kwargs)
    model = DistrQLearning(env=env, gamma=float(mdl["gamma"]), epsilon=float(mdl["epsilon"]),
                           epsilon_decay_rate=float(mdl["epsilon_decay_rate"]), lr=float(mdl["lr"]),
                           lr_decay_rate=float(mdl["lr_decay_rate"]), default_q=float(mdl["default_q"]), seed=seed)
    num_episodes = int(mdl["num_episodes"])
    model.learn(num_episodes=num_episodes, out_dir=out_dir, checkpoint_freq=int(misc["checkpoint_freq"]),
                exploit_freq=int(misc["exploit_freq"]))
    model.save(os.path.join(out_dir, "distr_q_model.pkl"))
    elapsed_time = time.time() - start_time
    print("DONE!")                                                       # main.py:68-78
    print(f"TOTAL TIME: {elapsed_time:.1f} seconds")
    print(f"Seconds per episode: {elapsed_time / max(num_episodes, 1):.1f}")
    print(f"Flatland step time: {env.flatland_step_time:.1f} seconds")
    print(f"Total step time: {env.step_time:.1f} seconds")
    print(f"Total last time: {env.last_time:.1f} seconds")
    print(f"Action selection time: {env.action_selection_time:.1f} seconds")
    print(f"Update time: {env.update_time:.1f} seconds")
    print(f"Flatland reset time: {env.reset_time:.1f} seconds")
    print(f"Total reset time: {env.reset_total_time:.1f} seconds")
    return model


def launch_grid(hyperparams: Dict[str, Sequence[float]], random_seeds: Sequence[int], out_dir: str, env_section: Dict[str, object],
                num_episodes: int, checkpoint_freq: int, exploit_freq: Optional[int], gamma: float = 1.0, default_q: float = 0.0,
                device: Optional[str] = None, q_cap: Optional[int] = None, env_cls=ASyncSwitchEnv, _engine_kwargs=None,
                rng: str = "philox", malfunction_rng: str = "philox") -> List[str]:
    """hyperparam_tuning.py:42-91: every (grid point, seed) pair gets ``out_dir/exp_i/seed_j/`` with its config.ini
    and the reference's output files.  One seed = one map (the generators are seeded with it), so each seed is ONE
    batched engine whose environments are the grid points; under torchrun the seeds are sharded over the ranks.
    With ``rng="reference"`` every environment learns on the reference's stream of its seed: environment i of a seed is
    the reference's main.py run for that (grid point, seed) -- on maps with malfunctions together with
    ``malfunction_rng="reference"`` (flatland's own malfunction stream of the seed)."""
    names = list(hyperparams)
    points = [dict(zip(names, v)) for v in product(*[hyperparams[n] for n in names])]
    rank, world_size, _ = sharding.world()
    device = device or default_device()
    lo, hi = sharding.shard_range(len(random_seeds), rank, world_size)
    written = []
    runs = []
    for rdx in range(lo, hi):
        seed = int(random_seeds[rdx])
        fx = fixture_from_env_section({k: str(v) for k, v in env_section.items()}, seed)
        mf = ParamMalfunctionGen(MalfunctionParameters(float(env_section.get("malfunction_rate", 0.0)),
                                                       int(env_section.get("min_duration", 0)), int(env_section.get("max_duration", 0))))
        env = env_cls(RailEnv(fx, malfunction_generator=mf), render_mode=None, max_steps=100_000, n_envs=len(points),
                      device=device, q_cap=q_cap, rng=rng, malfunction_rng=malfunction_rng, _engine_kwargs=_engine_kwargs)
        col = lambda k, d: np.array([p.get(k, d) for p in points], np.float64)
        model = DistrQLearning(env=env, gamma=gamma, epsilon=col("epsilon", 0.4), epsilon_decay_rate=col("epsilon_decay_rate", 0.0),
                               lr=col("lr", 0.4), lr_decay_rate=col("lr_decay_rate", 0.0), default_q=default_q,
                               seeds=np.full(len(points), seed, np.uint64))          # same seed for every point, as the reference
        runs.append((rdx, seed, model))
    # hyperparam_tuning.py:85-91 starts every run at once; here the seeds of this rank learn concurrently, one stream each
    learn_concurrently([m for _, _, m in runs], num_episodes, None, checkpoint_freq, exploit_freq)
    for rdx, seed, model in runs:
        for idx, params in enumerate(points):
            exp_dir = os.path.join(out_dir, f"exp_{idx}", f"seed_{rdx}")
            os.makedirs(exp_dir, exist_ok=True)
            config = configparser.ConfigParser()
            config["MISC"] = {"random_seed": str(seed), "out_dir": exp_dir, "checkpoint_freq": str(checkpoint_freq),
                              "exploit_freq": str(exploit_freq)}
            if rng != "philox":
                config["MISC"]["rng"] = rng
            if malfunction_rng != "philox":
                config["MISC"]["malfunction_rng"] = malfunction_rng
            config["ENV"] = {k: str(v) for k, v in env_section.items()}
            config["MODEL"] = {"gamma": str(gamma), **{k: str(params[k]) for k in names}, "default_q": str(default_q),
                               "num_episodes": str(num_episodes)}
            with open(os.path.join(exp_dir, "config.ini"), "w") as f:
                config.write(f)
            model.write_outputs(idx, exp_dir, exploit=exploit_freq is not None)
            written.append(exp_dir)
        model.env.engine.close()
    return written


def launch_eval(exp_dir_list: Sequence[str], distr_q_model_name: str = "distr_q_model.pkl", device: Optional[str] = None,
                q_cap: Optional[int] = None, env_cls=ASyncSwitchEnv, _engine_kwargs=None, num_evals: Optional[int] = None) -> Dict[str, np.ndarray]:
    """eval.py:31-97: for every experiment directory reload ``config.ini`` + the pickled Q-table and run the greedy
    ``test()`` -- once, or ten times when the map has malfunctions (eval.py:88); ``num_evals`` runs instead when given.
    The evaluations are the environments of one evaluation engine that reads the table once for all of them
    (``DistrQLearning.evaluate``); environment i draws its malfunctions from seed + i.  The first ten go to ``eval_i/`` like
    the reference's; with more than ten, ``eval_batched.npz`` holds every run."""
    out = {}
    device = device or default_device()
    for exp_dir in exp_dir_list:
        print(f"Evaluating {exp_dir}")
        config = configparser.ConfigParser()
        config.read(os.path.join(exp_dir, "config.ini"))
        envs, mdl, seed = config["ENV"], config["MODEL"], int(config["MISC"]["random_seed"])
        rate = float(envs["malfunction_rate"])
        mf = ParamMalfunctionGen(MalfunctionParameters(rate, int(envs["min_duration"]), int(envs["max_duration"])))
        n = int(num_evals) if num_evals is not None else (10 if rate > 0 else 1)
        cap = q_cap if q_cap is not None else (int(config["MISC"]["q_cap"]) if config["MISC"].get("q_cap") else None)
        # the learner's own engine only carries the map: one environment
        env = env_cls(RailEnv(fixture_from_env_section(dict(envs), seed), malfunction_generator=mf), render_mode=None,
                      max_steps=100_000, n_envs=1, device=device, q_cap=cap, _engine_kwargs=_engine_kwargs)
        model = DistrQLearning(env=env, gamma=float(mdl["gamma"]), epsilon=float(mdl["epsilon"]),
                               epsilon_decay_rate=float(mdl["epsilon_decay_rate"]), lr=float(mdl["lr"]),
                               lr_decay_rate=float(mdl["lr_decay_rate"]), default_q=float(mdl["default_q"]), seed=seed)
        cum, arrived, delays, _, _ = model.evaluate(read_q_table(os.path.join(exp_dir, distr_q_model_name)), n_runs=n,
                                                    out_dir=exp_dir if n > 10 else None)
        for i in range(min(n, 10)):
            print(f"Eval {i+1}")
            d = os.path.join(exp_dir, f"eval_{i}")
            os.makedirs(d, exist_ok=True)
            np.savez_compressed(os.path.join(d, "cum_reward.npz"), x=cum[i])                 # distr_q.py:237-239
            np.savez_compressed(os.path.join(d, "delays.npz"), x=list(delays[i]))
        out[exp_dir] = np.stack([cum, arrived])
        env.engine.close()
    return out


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("-c", "--config", type=str, help="Config file path (required unless --eval)")
    ap.add_argument("--eval", nargs="+", metavar="EXP_DIR", default=None,
                    help="evaluate the distr_q_model.pkl of these experiment directories (eval.py) instead of learning")
    ap.add_argument("--num-evals", type=int, default=None,
                    help="--eval: greedy runs per experiment, seeds random_seed + i (default: 10 on maps with malfunctions, else 1)")
    ap.add_argument("--device", default=None, help="default: cuda:<LOCAL_RANK>")
    ap.add_argument("--q-cap", type=int, default=None, help="Q hash rows per environment (default: MISC.q_cap, else sized from the map)")
    ap.add_argument("--rng", choices=("philox", "reference"), default=None,
                    help="epsilon-greedy stream of learn(): philox, or the reference's own numpy stream (default: MISC.rng, else philox)")
    ap.add_argument("--malfunction-rng", choices=("philox", "reference"), default=None,
                    help="malfunction draws: philox, or flatland's own numpy stream of the seed (default: MISC.malfunction_rng, else philox)")
    args = ap.parse_args(argv)
    if args.eval:
        launch_eval(args.eval, device=args.device, q_cap=args.q_cap, num_evals=args.num_evals)
        return
    if not args.config:
        ap.error("the following arguments are required: -c/--config")
    launch_experiment(args.config, device=args.device, q_cap=args.q_cap, rng=args.rng, malfunction_rng=args.malfunction_rng)


if __name__ == "__main__":
    main()
