"""Drop-in surface: the two classes main.py / test_model.py / eval.py / hyperparam_tuning.py construct
(SURVEY.md section 8b), batched over B lockstep environments on one GPU.

    rail_env = RailEnv(fixture)                                   # replaces main.py:36-49 (flatland generators)
    env      = ASyncSwitchEnv(rail_env, max_steps=100_000, n_envs=4096)          # main.py:51
    model    = DistrQLearning(env=env, gamma=1., epsilon=.5, ..., seed=450565)   # main.py:53-60
    model.learn(num_episodes, out_dir, checkpoint_freq, exploit_freq)            # main.py:63
    model.save(os.path.join(out_dir, "distr_q_model.pkl"))                       # main.py:66

Environment ``i`` is an independent learner with seed ``seed + i`` (hyperparam_tuning.py's process fan-out
becomes the env axis; per-env hyper-parameter arrays give the grid).  The decision loop itself
(distr_q.py:302-362) runs inside the CUDA kernel; the host only launches chunks and collects metrics.
Outputs keep the reference's file names and dict layout (distr_q.py:288-294, 368-375, 521-523).
"""
from __future__ import annotations

import os
import pickle
import queue
import threading
import time
from typing import Dict, Iterator, List, Optional, Sequence

import numpy as np

from .backend import MODE_GREEDY, MODE_LEARN, Engine, RailMap, train_set


class Discrete:
    """gymnasium.spaces.Discrete as the reference uses it (switch_agents.py:204-259, distr_q.py:316-317):
    ``n``, ``contains``, ``seed`` and ``sample(mask)`` = ``Generator(PCG64(seed)).choice(where(mask))``."""

    def __init__(self, n: int):
        self.n = int(n)
        self._rng = np.random.default_rng()

    def contains(self, x) -> bool:
        return isinstance(x, (int, np.integer)) and 0 <= int(x) < self.n

    def seed(self, seed=None):
        self._rng = np.random.default_rng(seed)

    def sample(self, mask=None) -> int:
        if mask is None:
            return int(self._rng.integers(self.n))
        valid = np.where(np.asarray(mask) == 1)[0]
        return int(self._rng.choice(valid)) if len(valid) else 0


class MalfunctionParameters:
    """flatland.envs.malfunction_generators.MalfunctionParameters (main.py:28-32)."""

    def __init__(self, malfunction_rate=0.0, min_duration=0, max_duration=0):
        self.malfunction_rate, self.min_duration, self.max_duration = malfunction_rate, min_duration, max_duration


class ParamMalfunctionGen:
    def __init__(self, parameters: MalfunctionParameters):
        self.parameters = parameters


class RailEnv:
    """Fixture-backed stand-in for the flatland RailEnv constructor lines (main.py:36-49): the map, line
    and timetable come from a fixture dict / .npz (see mapgen.py) instead of the flatland generators."""

    def __init__(self, fixture, malfunction_generator=None, **_ignored):
        if isinstance(fixture, str):
            from .mapgen import load_fixture
            fixture = load_fixture(fixture)
        self.fixture = dict(fixture)
        if malfunction_generator is not None:
            p = getattr(malfunction_generator, "parameters", malfunction_generator)
            self.fixture["malfunction_rate"] = float(p.malfunction_rate)
            self.fixture["min_duration"] = int(p.min_duration)
            self.fixture["max_duration"] = int(p.max_duration)
        self.height, self.width = self.fixture["grid"].shape
        self._elapsed_steps = 0

    def get_num_agents(self) -> int:
        return len(self.fixture["init_dir"])


def default_q_cap(rail_map: RailMap) -> int:
    """Q hash rows per environment when the caller gives none: the next power of two above twice the states one learner
    can reach -- every optimistic row of distr_q.py:81-181 (load() imports all of them) plus, per (port, target) pair that
    occurs, the 15 x 3 semaphore / delay variants the trains actually standing there can produce; capped so that the
    state stays allocatable.  A table that still fills up is reported (SFL_ERR_Q_FULL), never silently wrong."""
    t, tr = rail_map.tab, rail_map.trains
    init_rows = int((np.asarray(tr.qinit_act) >= 0).sum()) * 45
    reach = int(t.NP) * min(len(tr.targets), 4) * 12
    want = 2 * (init_rows + reach) + 256
    cap = 1024
    while cap < want and cap < (1 << 20):
        cap *= 2
    return cap


class ASyncSwitchEnv:
    """Batched counterpart of switch_env.py:605-678.  Holds the map tables and the engine; the AEC
    per-decision protocol (agent_iter / last / step) is executed on the device by the learner's kernel."""

    engine_cls = Engine

    def __init__(self, rail_env: RailEnv, max_steps: int = 200, render_mode=None, observer=None, seed=None,
                 n_envs: int = 1, device: str = "cuda:0", q_cap: Optional[int] = None, ep_cap: int = 128, shared_q: bool = False,
                 phase_timers: bool = False, rng: str = "philox", malfunction_rng: str = "philox", _engine_kwargs=None):
        """``phase_timers``: run the instrumented kernel (per-phase cycle counters, a few per cent slower) so that all seven
        wall-clock accumulators of switch_env.py:67-73 are filled; without it the fused kernel books its whole time on
        ``step_time`` (and resets on ``reset_total_time``).
        ``rng="reference"``: learn() draws its epsilon-greedy choices from the reference's own numpy stream
        (``np.random.default_rng(seed)`` per learn() call, distr_q.py:269, 315-317), so environment i with seed s makes the
        decisions of the reference's learn() with seed s -- on maps with malfunctions together with
        ``malfunction_rng="reference"``.  "philox" (default): the faster counter-based stream.
        ``malfunction_rng="reference"``: the malfunctions come from flatland's own stream, ``np.random.RandomState(seed)``
        created by every episode's ``rail_env.reset(random_seed=seed)`` (switch_env.py:99): environment i with seed s has
        the malfunctions of the reference's episodes with seed s, in learn(), test() and the AEC protocol (whose
        ``reset()`` then needs an explicit seed).  "philox" (default): the counter-based draws."""
        self.rail_env = rail_env
        self.max_steps = max_steps
        self.render_mode = render_mode
        self.seed = seed
        self.n_envs = int(n_envs)
        kw = dict(act_cap=1, shared_q=shared_q, phase_clock=bool(phase_timers), rng=rng, malfunction_rng=malfunction_rng)
        kw.update(_engine_kwargs or {})
        self.rail_map = RailMap(rail_env.fixture, device_bfs=self.engine_cls.bfs_device(device))
        self.possible_agents = self.rail_map.tab.switch_names()          # switch_env.py:51-52
        self.agents = self.possible_agents
        if q_cap is None:
            q_cap = 2 if shared_q else default_q_cap(self.rail_map)
        self.engine = self.engine_cls(self.rail_map, n_envs=self.n_envs, device=device, q_cap=q_cap, max_steps=max_steps, ep_cap=ep_cap, **kw)
        # the seven wall-clock accumulators main.py:72-78 prints (switch_env.py:67-73); the device loop has no
        # per-phase split, so the kernel time is booked on step_time and resets on reset_total_time
        self.flatland_step_time = self.step_time = self.last_time = 0.0
        self.action_selection_time = self.update_time = self.reset_time = self.reset_total_time = 0.0
        self.num_malfunctions = 0
        self.train_to_last_node: Dict[int, tuple] = {}
        self._spaces: Dict[str, Discrete] = {}
        self._rec = None
        self._aec_hparams = None
        self.view = 0
        self.agent_selection, self.active_train = None, None
        self.terminated = self.truncated = False

    def action_space_n(self, agent: str) -> int:
        return int(self.rail_map.tab.sw_A[self.agents.index(agent)])

    def action_space(self, agent: str) -> Discrete:                       # switch_env.py:85-91
        sp = self._spaces.get(agent)
        if sp is None:
            sp = self._spaces[agent] = Discrete(self.action_space_n(agent))
        return sp

    # ------------------------------------------------------------------ the AEC protocol, host-driven (switch_env.py:93-158, 616-678)
    # One kernel launch per step(): the chosen action is applied on the device, the trains advance to the next decision
    # point, and the next (switch, train) with its observation comes back.  With n_envs > 1 every call handles all
    # environments in lockstep (``last_batch`` / ``step_batch``); the reference-shaped calls below address environment
    # ``view`` (0) and need n_envs == 1 for ``step``.
    def reset(self, seed=None, options=None):
        eng = self.engine
        if seed is None and eng.malfunction_rng == "reference":
            # the reference would continue flatland's stream (or seed it from entropy), which this mode does not model
            raise ValueError('reset() with malfunction_rng="reference" needs an explicit seed: reset(seed=...)')
        if seed is not None:
            self.seed = seed
        base = 0 if self.seed is None else int(self.seed)
        hp = self._aec_hparams or {}
        eng.set_hparams(**hp, seeds=np.arange(self.n_envs, dtype=np.uint64) + np.uint64(base), episodes=1)
        t0 = time.time()
        eng.reset(keep_q=True, keep_interactions=True)
        self._rec = eng.step(None)
        self.reset_total_time += time.time() - t0
        self._sync_view()

    def _sync_view(self):
        r = self._rec[self.view]
        self.terminated, self.truncated = bool(r["done"] & 1), bool(r["done"] & 2)
        self.rail_env._elapsed_steps = int(r["elapsed"])
        self.agent_selection = self.agents[int(r["sw"])] if r["pending"] else None
        self.active_train = int(r["train"]) if r["pending"] else None

    def agent_iter(self, max_iter: int = 2 ** 63):                        # switch_env.py:616-622
        n = 0
        while self._rec is not None and self._rec[self.view]["pending"] and n < max_iter:
            n += 1
            self._sync_view()
            yield self.agent_selection

    def observe(self, agent=None) -> np.ndarray:                          # switch_env.py:668-678 -> observer.py:246-308
        return np.array(self.rail_map.key_to_obs(int(self._rec[self.view]["key"])), dtype=np.int64)

    def last(self, observe: bool = True):
        """pettingzoo AECEnv.last(): (obs, rewards {train: float}, terminated, truncated, info)."""
        r = self._rec[self.view]
        T = self.rail_map.trains.T
        if not r["pending"]:
            return None, {h: 0.0 for h in range(T)}, self.terminated, self.truncated, {}
        A = self.action_space_n(self.agent_selection)
        mask = np.array([(int(r["mask"]) >> a) & 1 for a in range(A)], dtype=np.int8)
        rewards = {h: float(r["rewards"][h]) for h in range(T)}
        return (self.observe() if observe else None), rewards, self.terminated, self.truncated, \
            {"action_mask": mask, "active_train": int(r["train"])}

    def step(self, action):                                               # switch_env.py:632-666
        if self.n_envs != 1:
            raise RuntimeError("step() addresses one environment; use step_batch() with n_envs > 1")
        r = self._rec[self.view]
        if action is None or not r["pending"]:
            return {}
        if not self.action_space(self.agent_selection).contains(action):
            raise AssertionError(f"invalid action {action} for {self.agent_selection}")        # switch_env.py:213-215
        return self.step_batch([int(action)])[0]

    def last_batch(self) -> np.ndarray:
        """The per-environment ``sfl_step_rec`` array (pending, sw, train, key, mask, done, elapsed, rewards...)."""
        return self._rec

    def step_batch(self, actions):
        t0 = time.time()
        self._rec = self.engine.step(actions)
        self.engine.check_errors(allow=1)
        self.step_time += time.time() - t0
        self._sync_view()
        cells = self.rail_map.tab.switch_cells
        out = []
        for r in self._rec:
            nxt = int(r["last_next_sw"])
            out.append({"next_switch": tuple(int(x) for x in cells[nxt]) if nxt >= 0 else None,
                        "arrived_trains": train_set(r["arrived"], r["arrived_hi"], self.rail_map.trains.T)})
        return out

    def close(self):
        pass


class _CheckpointWriter:
    """The thread that writes learn()'s checkpoint files while the next episodes run.  Each checkpoint fills one of two host
    staging buffers (``staging()`` waits while both are still being written) and hands the writer a job that reads it.
    ``overlap``: True runs the jobs on the thread, False in the caller at ``submit`` (a run that waits at every checkpoint),
    None: no checkpoints.  Leaving the ``with`` block waits for the jobs and re-raises the first exception of one; when the
    block itself raises (an error of learn(), KeyboardInterrupt), the jobs not yet started are dropped instead of written."""

    def __init__(self, overlap: Optional[bool]):
        self.free: "queue.Queue[dict]" = queue.Queue()
        for _ in range(2):
            self.free.put({})
        self.jobs: "queue.Queue" = queue.Queue()
        self.errors: List[BaseException] = []
        self.cancelled = False
        self.thread = threading.Thread(target=self._work, daemon=True) if overlap else None
        if self.thread is not None:
            self.thread.start()

    def staging(self) -> dict:
        return self.free.get()

    def submit(self, job, staging: dict):
        if self.errors:
            raise self.errors[0]
        if self.thread is not None:
            self.jobs.put((job, staging))
            return
        try:
            job()
        finally:
            self.free.put(staging)

    def _work(self):
        while True:
            item = self.jobs.get()
            if item is None:
                return
            job, staging = item
            try:
                if not self.errors and not self.cancelled:
                    job()
            except BaseException as ex:                # re-raised by submit() / __exit__ in learn()'s thread
                self.errors.append(ex)
            finally:
                self.free.put(staging)

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        self.cancelled = exc_type is not None
        if self.thread is not None:
            self.jobs.put(None)
            self.thread.join()
        if exc_type is None and self.errors:
            raise self.errors[0]
        return False


def _dump_q(q: Dict[tuple, List[float]], filename: str):
    """distr_q.py:521-523: pickle the table with np.int64 key elements (observer.py:306)."""
    q = {tuple(np.int64(x) for x in k): list(v) for k, v in q.items()}
    with open(filename, "wb") as f:
        pickle.dump(q, f)


class DistrQLearning:
    """Batched counterpart of distr_q.py:11-527."""

    _overlap_checkpoints = True              # False: learn() writes each checkpoint before it goes on (same files)

    def __init__(self, env: ASyncSwitchEnv, gamma=1.0, epsilon=0.4, epsilon_decay_rate=0.0, lr=0.4, lr_decay_rate=0.0,
                 default_q=0.0, seed=450565, seeds: Optional[Sequence[int]] = None, dist=None):
        self.env = env
        self.gamma, self.initial_epsilon, self.epsilon_decay_rate = gamma, epsilon, epsilon_decay_rate
        self.initial_lr, self.lr_decay_rate, self.default_q = lr, lr_decay_rate, default_q
        self.seed = seed
        self.seeds = (np.asarray(seeds, np.uint64) if seeds is not None
                      else np.arange(env.n_envs, dtype=np.uint64) + np.uint64(seed))
        self.ticks_per_launch = 512
        self.dist = dist                       # torch.distributed (initialised) for the shared-table all-reduce, else None
        self.primary_env = 0                 # the env whose curves / Q-table go to the reference-named files
        self._q_table: Dict[tuple, List[float]] = {}
        self._q_stale = False                # the device tables are newer than _q_table (learn() / test() ran)
        self.total_decisions = 0
        self._q_inited = False
        self._table_dirty = False            # device tables hold rows created before q-init (load() / test())
        self._stream_fresh = True

    @property
    def q_table(self) -> Dict[tuple, List[float]]:
        """The reference's ``q_table`` dict (distr_q.py:42) of the primary environment.  The tables live on the device;
        after ``learn()`` / ``test()`` the dict is read back on first use (``save()``, the host-side learner methods, ...)."""
        if self._q_stale:
            p = self.primary_env
            self._q_table = self.env.engine.export_q(p, include_init=self._q_inited, default_q=self._default_q_of(p))
            self._q_stale = False
        return self._q_table

    @q_table.setter
    def q_table(self, q):
        self._q_table, self._q_stale = q, False

    # ------------------------------------------------------------------ internals
    def _hparams(self, episodes: int, episode_base: int = 0):
        self.env.engine.set_hparams(gamma=self.gamma, epsilon=self.initial_epsilon, epsilon_decay_rate=self.epsilon_decay_rate,
                                    lr=self.initial_lr, lr_decay_rate=self.lr_decay_rate, default_q=self.default_q,
                                    seeds=self.seeds, episodes=episodes, episode_base=episode_base)

    def _begin_tables(self, keep_q: bool):
        """Shared-table mode (extension): the one table of this engine replaces the per-environment tables."""
        eng = self.env.engine
        if eng.shared_q and not keep_q:
            eng.init_shared_q(self._default_q_of(0), q_init=True)

    def _run_until_halted(self, mode: int) -> np.ndarray:
        eng = self.env.engine
        t0 = time.time()
        while True:
            if eng.shared_q and mode == MODE_LEARN:
                eng.run_shared(self.ticks_per_launch, self.dist)    # every ticks_per_launch ticks the mean TD steps are folded in
            else:
                eng.run(mode, self.ticks_per_launch)
            c = eng.counters()
            if c["err"].any():
                eng.check_errors()
            if (c["halted"] == 1).all():
                break
        if eng.shared_q and mode == MODE_LEARN:
            eng.shared_q_flush()
        dt = time.time() - t0
        self.env.step_time += dt
        if getattr(eng, "phase_clock", False):
            # switch_env.py:67-73: split the kernel time by the per-phase cycle counters of the instrumented kernel
            ph = c["phase_cycles"].astype(np.float64).sum(axis=0)
            if ph.sum() > 0:
                sh = ph / ph.sum()
                env = self.env
                env.flatland_step_time += dt * sh[0]; env.last_time += dt * sh[1]; env.action_selection_time += dt * sh[2]
                env.update_time += dt * sh[4]; env.reset_time += dt * sh[5]
        self.total_decisions += int(c["decisions"].sum())
        return c

    def _apply_q_init_to_existing_rows(self):
        """distr_q.py:156-158,179-181 ASSIGN the initial rows at t == 0, overwriting whatever an earlier learn() / load() /
        test() put there (on the device, for all environments at once)."""
        eng = self.env.engine
        if not eng.shared_q:
            eng.reapply_q_init()
            return
        q = eng.shared_q_table()                                          # shared-table mode: the one dense table, on the host
        tr = self.env.rail_map.trains
        port, tgt = np.nonzero(np.asarray(tr.qinit_act) >= 0)
        act, val = np.asarray(tr.qinit_act)[port, tgt], np.asarray(tr.qinit_val)[port, tgt]
        for semb in range(1, 16):
            q[port, tgt, semb, :, :] = self._default_q_of(0)
            q[port, tgt, semb, :, act] = val[:, None]
        eng._upload("shared_q", q)

    def learn_chunk(self, max_ticks: Optional[int] = None) -> np.ndarray:
        """Streaming API: upload the per-env hyper-parameter block, advance every environment by up to ``max_ticks``
        flatland ticks of learn() (no episode limit) and return the per-env counters (host array).
        bench.py times this call for its end-to-end number."""
        eng = self.env.engine
        if self._stream_fresh:
            self._hparams(-1)
            eng.reset()
            eng.enable_q_init(True)
            self._begin_tables(False)
            self._q_inited = True
            self._stream_fresh = False
        else:
            eng._upload("hparams", eng.hparams)
        if eng.shared_q:
            eng.run_shared(self.ticks_per_launch if max_ticks is None else max_ticks, self.dist)
        else:
            eng.run(MODE_LEARN, self.ticks_per_launch if max_ticks is None else max_ticks)
        return eng.counters()

    # ------------------------------------------------------------------ distr_q.py:244-379
    def learn(self, num_episodes: int, out_dir: Optional[str], checkpoint_freq: int, exploit_freq: Optional[int] = None,
              env_out_dirs: Optional[Sequence[str]] = None):
        """distr_q.py:244-379 for every environment at once.  ``out_dir`` gets the primary environment's files, as the
        reference's.  ``env_out_dirs``: one directory per environment, each of which also gets its environment's checkpoint
        files (checkpoint_N.pkl and the five *_checkpoint_N.npz of distr_q.py:288-294).  The checkpoints are written on a
        thread of their own from one device-side compaction of every table while the next episodes run; learn() waits for
        them before it returns and re-raises what failed there."""
        eng, env = self.env.engine, self.env
        B, T = env.n_envs, env.rail_map.trains.T
        p = self.primary_env
        if env_out_dirs is not None and len(env_out_dirs) != B:
            raise ValueError(f"env_out_dirs has {len(env_out_dirs)} directories for {B} environments")
        targets = ([(p, out_dir)] if out_dir else []) + [(i, d) for i, d in enumerate(env_out_dirs or [])]
        for _, d in targets:
            os.makedirs(d, exist_ok=True)
        cum_reward = np.zeros((B, num_episodes))
        arrived = np.zeros((B, num_episodes), np.int32)
        delays = np.zeros((B, num_episodes, T))
        num_malf = np.zeros((B, num_episodes), np.int32)
        cum_reward_exploit, arrived_exploit = [], []
        t_start = time.time()
        # pause points: the reference exploits / checkpoints BEFORE episode t when (t+1) % freq == 0 (distr_q.py:278-294)
        pauses = sorted({t for t in range(num_episodes)
                         if (exploit_freq and (t + 1) % exploit_freq == 0) or (checkpoint_freq and (t + 1) % checkpoint_freq == 0)}
                        | {num_episodes})
        done, first = 0, True
        with _CheckpointWriter(self._overlap_checkpoints if targets and checkpoint_freq else None) as writer:
            for cut in pauses:
                while done < cut:                                   # run episodes [done, cut) in ep_cap-sized launches
                    seg = min(cut - done, eng.cfg.ep_cap)
                    self._hparams(seg, episode_base=done)
                    if first:
                        t0 = time.time()
                        eng.reset(keep_q=self._table_dirty, keep_interactions=False)     # agent_num_interactions is per learn() (:263)
                        self._begin_tables(self._table_dirty)
                        if self._table_dirty:
                            self._apply_q_init_to_existing_rows()
                        eng.enable_q_init(True)                                           # distr_q.py:299-300
                        self._q_inited = True
                        first = False
                        env.reset_total_time += time.time() - t0
                    else:
                        eng.reset(keep_q=True, keep_interactions=True)
                    self._run_until_halted(MODE_LEARN)
                    _, log, dl = eng.episode_log()
                    cum_reward[:, done:done + seg] = log["cum_reward"][:, :seg]
                    arrived[:, done:done + seg] = log["arrived"][:, :seg]
                    num_malf[:, done:done + seg] = log["num_malfunctions"][:, :seg]
                    last_mask = log[["arrived_mask", "arrived_mask_hi"]][:, seg - 1].copy()
                    delays[:, done:done + seg] = dl[:, :seg]
                    done += seg
                if cut >= num_episodes:
                    break
                if exploit_freq and (cut + 1) % exploit_freq == 0:
                    r, a, _ = self.test(out_dir=None, plot=False, save_outputs=False, _batched=True)
                    cum_reward_exploit.append(r)
                    arrived_exploit.append(a)
                if checkpoint_freq and (cut + 1) % checkpoint_freq == 0 and targets:
                    self._checkpoint(writer, targets, cut, cum_reward, arrived, delays, num_malf)
        self._table_dirty = True
        self._q_stale = True                 # q_table is read back from the device when it is next used
        at_dest = [train_set(mk["arrived_mask"], mk["arrived_mask_hi"], T) for mk in last_mask] if num_episodes else [[] for _ in range(B)]
        self.metrics = dict(cum_reward=cum_reward, arrived_trains=arrived, delays=delays, num_malfunctions=num_malf, trains_at_dest=at_dest,
                            cum_reward_exploit=np.array(cum_reward_exploit), arrived_trains_exploit=np.array(arrived_exploit),
                            wall_s=time.time() - t_start)
        if out_dir:
            self.write_outputs(p, out_dir, exploit=exploit_freq is not None, pkl=False)
            np.savez_compressed(os.path.join(out_dir, "batched_metrics.npz"), cum_reward=cum_reward, arrived_trains=arrived,
                                delays=delays, num_malfunctions=num_malf, seeds=self.seeds)
        if num_episodes:
            env.num_malfunctions = int(num_malf[p, -1])
            env.train_to_last_node = {h: (None, float(delays[p, -1, h])) for h in range(T)}
        env.close()

    def _checkpoint(self, writer: _CheckpointWriter, targets, cut: int, cum_reward, arrived, delays, num_malf):
        """distr_q.py:288-294 before episode ``cut`` for every (environment, directory) of ``targets``: the tables are
        compacted on the device and copied out behind the launches already queued; the writer turns them into the files.
        The metric rows [:cut] are final here, and cum_reward is zero from ``cut`` on, so the job reads them in place."""
        eng = self.env.engine
        envs = sorted({i for i, _ in targets})
        include_init, dq = self._q_inited, {i: self._default_q_of(i) for i in envs}
        staging = writer.staging()
        if eng.shared_q:
            shared = dict(zip(envs, eng.export_q_batch(envs, include_init, [dq[i] for i in envs])))
        else:
            snap = eng.compact_q(envs[0], envs[-1] + 1, staging)
        n_ep = cum_reward.shape[1]

        def job():
            init = {}
            if not eng.shared_q:
                snap.wait()
            # one table in memory at a time; the primary environment's is kept for its second directory only
            uses = {i: sum(1 for j, _ in targets if j == i) for i in envs}
            kept: Dict[int, Dict[tuple, List[float]]] = {}
            for i, d in targets:
                q = kept.pop(i, None)
                if q is None and eng.shared_q:
                    q = shared[i]
                elif q is None:
                    if include_init and dq[i] not in init:
                        init[dq[i]] = self.env.rail_map.q_init_rows(dq[i])
                    q = snap.table(i, init[dq[i]] if include_init else None)
                uses[i] -= 1
                if uses[i]:
                    kept[i] = q
                _dump_q(q, os.path.join(d, f"checkpoint_{cut + 1}.pkl"))
                del q
                np.savez_compressed(os.path.join(d, f"cum_reward_checkpoint_{cut + 1}.npz"),
                                    x=np.concatenate([cum_reward[i, :cut], np.zeros(n_ep - cut)]))
                np.savez_compressed(os.path.join(d, f"arrived_trains_checkpoint_{cut + 1}.npz"), x=arrived[i, :cut])
                np.savez_compressed(os.path.join(d, f"delays_checkpoint_{cut + 1}.npz"), x=delays[i, :cut])
                np.savez_compressed(os.path.join(d, f"trains_at_dest_checkpoint_{cut + 1}.npz"), x=[])   # SURVEY App. A #14
                np.savez_compressed(os.path.join(d, f"num_malfunctions_checkpoint_{cut + 1}.npz"), x=num_malf[i, :cut])

        writer.submit(job, staging)

    def env_q_tables(self, envs: Optional[Sequence[int]] = None) -> Iterator[Dict[tuple, List[float]]]:
        """The ``q_table`` of every environment of ``envs`` (consecutive indices, default all) -- the dicts ``save()``
        pickles for that environment -- from one compaction of their tables on the device, built one at a time in the
        order of ``envs`` (``Engine.iter_q_batch``), so that a caller writing them holds one table at a time."""
        envs = list(range(self.env.n_envs) if envs is None else envs)
        return self.env.engine.iter_q_batch(envs, include_init=self._q_inited, default_q=[self._default_q_of(i) for i in envs])

    def _default_q_of(self, i: int) -> float:
        d = np.asarray(self.default_q, np.float64).reshape(-1)
        return float(d[i % d.size])

    def write_outputs(self, env_index: int, out_dir: str, exploit: bool = True, pkl: bool = True,
                      q_table: Optional[Dict[tuple, List[float]]] = None):
        """The reference's end-of-learn files (distr_q.py:368-375, main.py:66) for environment ``env_index``.  ``q_table``:
        the environment's table when the caller has it already (``env_q_tables``), else it is exported here."""
        m, i = self.metrics, env_index
        os.makedirs(out_dir, exist_ok=True)
        np.savez_compressed(os.path.join(out_dir, "cum_reward.npz"), x=m["cum_reward"][i])
        np.savez_compressed(os.path.join(out_dir, "arrived_trains.npz"), x=m["arrived_trains"][i])
        np.savez_compressed(os.path.join(out_dir, "delays.npz"), x=m["delays"][i])
        np.savez_compressed(os.path.join(out_dir, "num_malfunctions.npz"), x=m["num_malfunctions"][i])
        np.savez_compressed(os.path.join(out_dir, "trains_at_dest.npz"), x=m["trains_at_dest"][i])     # distr_q.py:371
        if exploit:
            np.savez_compressed(os.path.join(out_dir, "cum_reward_exploit.npz"), x=[r[i] for r in m["cum_reward_exploit"]])
            np.savez_compressed(os.path.join(out_dir, "arrived_trains_exploit.npz"), x=[a[i] for a in m["arrived_trains_exploit"]])
        if pkl and q_table is not None:
            _dump_q(q_table, os.path.join(out_dir, "distr_q_model.pkl"))
        elif pkl:
            keep = self.q_table
            self.q_table = self.env.engine.export_q(i, include_init=self._q_inited, default_q=self._default_q_of(i))
            self.save(os.path.join(out_dir, "distr_q_model.pkl"))
            self.q_table = keep

    # ------------------------------------------------------------------ distr_q.py:184-241
    def test(self, out_dir, plot=False, save_outputs=True, _batched=False):
        """Greedy rollout of every environment (one episode each); returns env 0's (cum_reward, arrived, delays)
        like the reference unless ``_batched``."""
        eng, env = self.env.engine, self.env
        T = env.rail_map.trains.T
        self._hparams(1)
        eng.reset(keep_q=True, keep_interactions=True)
        eng.enable_q_init(self._q_inited)
        self._run_until_halted(MODE_GREEDY)
        self._table_dirty = True
        _, log, dl = eng.episode_log()
        cum, arr, delays = log["cum_reward"][:, 0].copy(), log["arrived"][:, 0].copy(), dl[:, 0].astype(np.float64)
        p = self.primary_env
        if save_outputs:
            print(f"Terminated in {int(log['decisions'][p, 0])} steps ({int(log['ticks'][p, 0])} flatland steps), "
                  f"cumulative reward = {cum[p]}")
            print(f"Arrived trains: {int(arr[p])} / {T}")
            print(f"Delays: {list(delays[p])}")
            print(f"Num malfunctions: {int(log['num_malfunctions'][p, 0])}")
            if out_dir:
                np.savez_compressed(os.path.join(out_dir, "cum_reward.npz"), x=cum[p])
                np.savez_compressed(os.path.join(out_dir, "delays.npz"), x=list(delays[p]))
        if _batched:
            return cum, arr, delays
        self._q_stale = True                 # test() inserts rows (App. A #15)
        return float(cum[p]), int(arr[p]), list(delays[p])

    # ------------------------------------------------------------------ evaluation on one read-only table (extension)
    def evaluate(self, q_table: Optional[Dict[tuple, List[float]]] = None, n_runs: Optional[int] = None,
                 seeds: Optional[Sequence[int]] = None, out_dir: Optional[str] = None):
        """Greedy rollouts of one table -- what eval.py does with ``load()`` + ``test()`` ten times -- on as many environments
        as wanted: one episode per environment of an evaluation engine on the same map (``Engine(eval_q=True)``), every
        environment reading the one read-only table.  ``q_table``: default ``self.q_table`` (with the optimistic rows when
        this learner was q-initialised).  ``seeds``: one per run; default ``seed + i`` for ``n_runs`` runs (default: as many
        as this learner has environments), the seeds ``test()`` gives its environments.

        Decisions and metrics equal ``load()`` + ``test()``; the one difference is that the table is not mutated: ``test()``
        inserts a default row at every lookup that misses (distr_q.py:482 -> :56-57), which never changes a decision.
        This learner's engine and tables are not touched.  Returns (cum_reward[n], arrived[n], delays[n, T],
        num_malfunctions[n], the arrived trains of every run); ``out_dir``: also writes them to ``eval_batched.npz``."""
        env = self.env
        q = self.q_table if q_table is None else q_table
        if seeds is None:
            n = env.n_envs if n_runs is None else int(n_runs)
            seeds = np.arange(n, dtype=np.uint64) + np.uint64(self.seed)
        seeds = np.asarray(seeds, np.uint64).reshape(-1)
        if n_runs is not None and len(seeds) != int(n_runs):
            raise ValueError(f"{len(seeds)} seeds for {n_runs} runs")
        n, T = len(seeds), env.rail_map.trains.T
        cap = 1024
        while cap < 2 * len(q) + 2:                                       # load factor at most one half
            cap *= 2
        learner = env.engine
        eng = env.engine_cls(env.rail_map, n_envs=n, device=learner.device, q_cap=cap, max_steps=env.max_steps, ep_cap=1,
                             eval_q=True, malfunction_rng=learner.malfunction_rng)
        try:
            eng.set_hparams(default_q=self._default_q_of(self.primary_env), seeds=seeds, episodes=1)
            eng.reset()
            eng.set_eval_table(q)
            t0 = time.time()
            while True:
                eng.run(MODE_GREEDY, self.ticks_per_launch)
                c = eng.counters()
                if c["err"].any():
                    eng.check_errors()
                if (c["halted"] == 1).all():
                    break
            self.eval_time = time.time() - t0
            _, log, dl = eng.episode_log()
        finally:
            eng.close()
        cum, arr = log["cum_reward"][:, 0].copy(), log["arrived"][:, 0].copy()
        delays, malf = dl[:, 0].astype(np.float64), log["num_malfunctions"][:, 0].copy()
        at_dest = [train_set(r["arrived_mask"], r["arrived_mask_hi"], T) for r in log[:, 0]]
        if out_dir:
            os.makedirs(out_dir, exist_ok=True)
            np.savez_compressed(os.path.join(out_dir, "eval_batched.npz"), cum_reward=cum, arrived_trains=arr, delays=delays,
                                num_malfunctions=malf, seeds=seeds,
                                arrived_mask=log["arrived_mask"][:, 0].copy(), arrived_mask_hi=log["arrived_mask_hi"][:, 0].copy())
        return cum, arr, delays, malf, at_dest

    # ------------------------------------------------------------------ distr_q.py:400-490, on the host dict
    # The reference's per-decision learner methods, for code that drives the AEC protocol itself (env.agent_iter /
    # last / step) and keeps the learning rule on the host.  They work on ``self.q_table`` exactly like the reference
    # (keys: observation tuples; rows: lists of floats; rows appear on first lookup); ``learn()`` / ``test()`` do the same
    # work on the device and overwrite ``q_table`` with the device tables when they finish.
    def _check_entry(self, state, agent) -> list:
        key = tuple(int(x) for x in state)
        row = self.q_table.get(key)
        if row is None:                                                    # distr_q.py:47-57
            row = self.q_table[key] = [self._default_q_of(self.primary_env)] * self.env.action_space(agent).n
        return row

    def eval(self, state, action, agent) -> float:                         # distr_q.py:400-417
        return self._check_entry(state, agent)[action]

    def max_q(self, state, agent) -> float:                                # distr_q.py:449-466 (ignores the action mask)
        if state is None:
            return 0.0
        return max(self._check_entry(state, agent))

    def max_action(self, state, agent, action_mask) -> int:                # distr_q.py:468-490
        row = self._check_entry(state, agent)
        best = int(np.argmax(row))
        if action_mask[best]:
            return best
        allowed = np.nonzero(action_mask)[0]
        return int(allowed[np.argmax(np.array(row)[allowed])])

    def update(self, state, action, reward, next_state, previous_agent, next_agent, agent_num_interactions):
        """distr_q.py:419-447: Q <- (1 - lr) Q + lr (r + gamma max_a' Q(s', a')), without the bootstrap when the train
        stayed at the same switch; lr = lr0 * lr_decay_rate ** (interactions of the previous switch)."""
        row = self._check_entry(state, previous_agent)
        lr0 = float(np.asarray(self.initial_lr, np.float64).reshape(-1)[0])
        decay = float(np.asarray(self.lr_decay_rate, np.float64).reshape(-1)[0])
        gamma = float(np.asarray(self.gamma, np.float64).reshape(-1)[0])
        lr = lr0 * (decay ** agent_num_interactions[previous_agent])
        if next_agent != previous_agent:
            row[action] = (1 - lr) * row[action] + lr * (reward + gamma * self.max_q(next_state, next_agent))
        else:
            row[action] = (1 - lr) * row[action] + lr * reward

    # ------------------------------------------------------------------ distr_q.py:492-527
    def save(self, filename: str, mode: str = "pickle"):
        if mode != "pickle":
            raise AttributeError("only mode='pickle' exists in the reference (distr_q.py:505-508 dispatch to undefined methods)")
        _dump_q(self.q_table, filename)

    def load(self, filename: str):
        self.q_table = read_q_table(filename)
        eng = self.env.engine
        if not eng.shared_q and len(self.q_table) >= eng.cfg.q_cap:
            raise ValueError(f"{filename}: {len(self.q_table)} rows do not fit the {eng.cfg.q_cap}-row Q tables of this env; "
                             f"construct ASyncSwitchEnv(q_cap=...) with a power of two above {2 * len(self.q_table)}")
        self._hparams(-1)
        eng.reset()
        for i in range(self.env.n_envs):
            eng.import_q(i, self.q_table)
        self._table_dirty = True
        self._q_inited = False


def read_q_table(filename: str) -> Dict[tuple, List[float]]:
    """A pickled q_table (distr_q_model.pkl / checkpoint_N.pkl, distr_q.py:521-527) as the dict ``load()`` keeps."""
    with open(filename, "rb") as f:
        q = pickle.load(f)
    return {tuple(int(x) for x in k): [float(x) for x in v] for k, v in q.items()}


def learn_concurrently(models: Sequence[DistrQLearning], num_episodes: int, out_dirs: Optional[Sequence[Optional[str]]] = None,
                       checkpoint_freq: int = 0, exploit_freq: Optional[int] = None,
                       env_out_dirs: Optional[Sequence[Optional[Sequence[str]]]] = None) -> None:
    """``learn()`` of several independent learners (different maps / seeds) at the same time on one GPU: one host thread and
    one CUDA stream per learner, so that their kernel launches overlap.  This is hyperparam_tuning.py:85-91 -- every
    (point, seed) run started at once, no communication -- with streams in place of OS processes; the results are those of
    calling ``learn()`` on each model in turn.  ``env_out_dirs``: one ``learn(env_out_dirs=...)`` list per model."""
    import torch
    out_dirs = list(out_dirs) if out_dirs is not None else [None] * len(models)
    env_out_dirs = list(env_out_dirs) if env_out_dirs is not None else [None] * len(models)
    if torch.cuda.is_available():
        torch.cuda.synchronize()                       # buffers were created on the default stream
    errors: List[BaseException] = []

    def work(m: DistrQLearning, out_dir: Optional[str], dirs: Optional[Sequence[str]]):
        try:
            dev = m.env.engine.device
            if dev.type == "cuda":
                stream = torch.cuda.Stream(device=dev)
                with torch.cuda.device(dev), torch.cuda.stream(stream):
                    m.learn(num_episodes, out_dir, checkpoint_freq, exploit_freq, env_out_dirs=dirs)
                    stream.synchronize()
            else:
                m.learn(num_episodes, out_dir, checkpoint_freq, exploit_freq, env_out_dirs=dirs)
        except BaseException as ex:                    # re-raised in the caller's thread
            errors.append(ex)

    threads = [threading.Thread(target=work, args=(m, d, e)) for m, d, e in zip(models, out_dirs, env_out_dirs)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
