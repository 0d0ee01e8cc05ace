"""Flatland's malfunction stream on the device (``Engine(malfunction_rng="reference")``, SFL_MALF_REFERENCE).

flatland's ``rail_env.reset(random_seed=seed)`` creates ``np.random.RandomState(seed)`` at every episode; every tick, for
every train in handle order, ``ParamMalfunctionGen.generate`` draws ``rand() < 1 - exp(-rate)`` and, on a hit,
``randint(min, max + 1) + 1`` steps (oracle/trainsim.py).  The engine generates that schedule on the device from the seed
alone, so seeded runs have the reference's malfunctions without a recorded schedule: the schedule is checked against
numpy, the goldens are reproduced from their seeds alone, and free-running learn(), test() and the AEC protocol against the
oracle.  CPU tests run the host build of the device sources (tests/emul); ``-m gpu`` the CUDA kernels at every lane width."""
import configparser
import ctypes as C
import math
import os
import pickle
import tempfile

import numpy as np
import pytest

from switchfl_b200 import api, backend, cli
from tests._parity import compare_trace, golden_events
from tests._util import golden_names, hparams, load_golden, q_dict
from tests.emulated import EmulEngine, EmulSwitchEnv, build_emul, emul_library
from tests.test_reference_stream import HP, I32MAX, golden_draws, many_train_map, oracle_learn, oracle_learn_call

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATES = (0.0, 1e-4, 0.01, 0.5, 5.0)
DURATIONS = ((5, 5), (0, 0), (2, 6), (5, 15), (0, 1023), (0, 1024), (0, 100000))
MALF_GOLDENS = [n for n in golden_names() if float(load_golden(n)[0]["malfunction_rate"]) > 0]


@pytest.fixture(scope="module")
def lib():
    return emul_library()


def gpu_engine(*a, **kw):
    return backend.Engine(*a, **kw)


def numpy_schedule(seed, rate, lo, hi, T, steps):
    """flatland's draws (trainsim.ParamMalfunctionGen.generate) for ticks 1 .. steps, every train, as a plain numpy loop."""
    p = 0.0 if rate <= 0 else 1.0 - math.exp(-rate)
    r = np.random.RandomState(seed)
    out = []
    for tick in range(1, steps + 1):
        for t in range(T):
            if r.rand() < p:
                out.append((tick, t, int(r.randint(lo, hi + 1)) + 1))
    return np.array(out, np.int32).reshape(-1, 3)


def applied_events(schedule, T, ticks):
    """The events an episode of ``ticks`` ticks applies: a draw takes effect only while the train's counter is 0, and every
    counter counts down once per tick (trainsim.RailEnv.step)."""
    by_tick = {}
    for tick, t, d in schedule:
        by_tick.setdefault(int(tick), []).append((int(t), int(d)))
    counter, out = [0] * T, []
    for tick in range(1, ticks + 1):
        for t, d in by_tick.get(tick, []):
            if counter[t] == 0 and d > 0:
                counter[t] = d
                out.append((tick, t, d))
        counter = [max(c - 1, 0) for c in counter]
    return out


# ---------------------------------------------------------------------------------------------- the schedule vs numpy
def schedule_seeds(k, n_random=30):
    r = np.random.default_rng(1000 + k)
    return [0, 1, 450565, I32MAX, 2 ** 32 - 1] + [int(x) for x in r.integers(0, 2 ** 32, n_random)]


def check_schedules(factory, **kw):
    """About 1200 (seed, rate, durations) triples on a map whose episodes are long enough that the draws cross several
    twists of the 624-word state; rate 5 makes most draws hits, so the randint words cross twists too."""
    fx, _ = load_golden("c1_synth18")
    fx = dict(fx, max_episode_steps=400)
    rm = backend.RailMap(fx)
    T, steps = rm.trains.T, 400
    k = 0
    for rate in RATES:
        for lo, hi in DURATIONS:
            seeds = schedule_seeds(k)
            k += 1
            eng = factory(rm, n_envs=len(seeds), q_cap=64, ep_cap=1, malfunction_rng="reference", ev_cap=T * steps, **kw)
            eng.set_hparams(**HP, seeds=seeds, malfunction_rate=rate, min_duration=lo, max_duration=hi)
            eng.reset()
            longest = 0
            for i, sd in enumerate(seeds):
                want = numpy_schedule(sd, rate, lo, hi, T, steps)
                got = eng.malfunction_schedule(i)
                assert np.array_equal(got, want), (rate, lo, hi, sd, len(got), len(want))
                longest = max(longest, len(want))
            assert eng.max_malfunction_events == longest
            if rate >= 0.5:
                assert longest > T * steps // 3
            eng.close()


def test_emul_schedule_matches_numpy():
    build_emul()
    check_schedules(EmulEngine)


def shipped_rates():
    from switchfl_b200 import mapgen
    rates = {float(load_golden(n)[0]["malfunction_rate"]) for n in golden_names()}
    rates |= {float(mapgen.c4_fixture()["malfunction_rate"]), float(mapgen.t100_fixture()["malfunction_rate"])}
    rates |= {float(many_train_map(n).fixture["malfunction_rate"]) for n in ("t65", "t100", "t128")}
    return sorted(rates | set(RATES) | {0.03, 0.02})


def test_hit_threshold_is_flatlands_comparison():
    """ceil(p 2^53) on the host with trainsim's p: a 53-bit draw k hits (rand() = k 2^-53 < p) iff k < the threshold."""
    from oracle.trainsim import MalfunctionParameters, ParamMalfunctionGen
    for rate in shipped_rates():
        p = ParamMalfunctionGen(MalfunctionParameters(rate, 0, 0)).prob()
        thr = backend.malf_hit_below(rate)
        assert thr == math.ceil(p * 2.0 ** 53)
        assert not (thr * 2.0 ** -53 < p), rate
        if thr:
            assert (thr - 1) * 2.0 ** -53 < p, rate


def check_refusals(factory):
    fx, _ = load_golden("slips24_t6")
    rm = backend.RailMap(fx)
    eng = factory(rm, n_envs=2, q_cap=64, malfunction_rng="reference")
    eng.set_hparams(**HP, seeds=[1, 2 ** 32])
    with pytest.raises(RuntimeError, match=r"Seed must be between 0 and 2\*\*32 - 1"):
        eng.reset()
    eng.set_hparams(**HP, seeds=[1, 2 ** 32 - 1], min_duration=6, max_duration=2)
    with pytest.raises(RuntimeError, match="min_duration > max_duration"):
        eng.reset()
    with pytest.raises(ValueError, match="set_replay"):
        eng.set_replay(None, [np.zeros((0, 3), np.int32)] * 2)
    eng.close()
    small = factory(rm, n_envs=2, q_cap=64, malfunction_rng="reference", ev_cap=3)
    small.set_hparams(**HP, seeds=[5, 6], malfunction_rate=0.5)
    with pytest.raises(RuntimeError, match="does not fit replay_ev"):
        small.reset()
    assert small.max_malfunction_events > 3
    small.close()


def test_emul_refusals(lib):
    build_emul()
    check_refusals(EmulEngine)
    fx, _ = load_golden("c1_synth18")
    rm = backend.RailMap(fx)
    with pytest.raises(ValueError, match="malfunction_rng must be one of"):
        EmulEngine(rm, n_envs=2, malfunction_rng="mt")
    with pytest.raises(RuntimeError, match="shared-table"):
        EmulEngine(rm, n_envs=2, q_cap=2, shared_q=True, malfunction_rng="reference")
    ctx = C.c_void_p()
    cfg = backend.Config(n_envs=2, q_cap=1024, pend_cap=8, max_steps=100, ep_cap=1, malf_rng=1)          # ev_cap 0
    assert lib.sfl_create(C.byref(rm.desc), C.byref(cfg), 0, C.byref(ctx)) == -1
    assert b"ev_cap >= 1" in lib.sfl_last_error()
    cfg = backend.Config(n_envs=2, q_cap=1024, pend_cap=8, max_steps=100, ep_cap=1, ev_cap=4, malf_rng=2)
    assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(backend.Sizes())) == -1
    assert b"malf_rng must be" in lib.sfl_last_error()
    eng = EmulEngine(rm, n_envs=1)
    with pytest.raises(RuntimeError, match="malfunction_schedule"):
        eng.malfunction_schedule(0)
    env = EmulSwitchEnv(api.RailEnv(fx), max_steps=100_000, q_cap=64, ep_cap=2, malfunction_rng="reference")
    with pytest.raises(ValueError, match="explicit seed"):
        env.reset()


@pytest.mark.parametrize("name", ("c1_synth18", "c4_rail100_t50"))
def test_sizes_and_launches_unchanged_without_the_option(lib, name):
    fx, _ = load_golden(name)
    rm = backend.RailMap(fx)
    sizes = {}
    for malf in (0, 1):
        cfg = backend.Config(n_envs=16, q_cap=1024, pend_cap=8, max_steps=100, dec_cap=4, ep_cap=2, ev_cap=8, malf_rng=malf)
        s = backend.Sizes()
        assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(s)) == 0
        sizes[malf] = {k: getattr(s, k) for k, _ in backend.Sizes._fields_}
    assert sizes[0] == sizes[1]                          # the schedule lives in replay_ev: no layout changes at all
    for mode in (backend.MODE_GREEDY, backend.MODE_REPLAY, backend.MODE_STEP):
        a = EmulEngine(rm, n_envs=16, ev_cap=8, act_cap=1, bind=False)
        b = EmulEngine(rm, n_envs=16, ev_cap=8, act_cap=1, bind=False, malfunction_rng="reference")
        assert a.describe_launch(mode) == b.describe_launch(mode)
    assert "KIND=learn" in a.describe_launch(backend.MODE_LEARN) and "KIND=full" in b.describe_launch(backend.MODE_LEARN)


# ---------------------------------------------------------------------------------------------- goldens from the seed alone
def check_golden_from_seed(name, factory, n_envs=2, lanes=None, chunk=None):
    """The reference's learn() from its seed alone: both streams on the device, no recorded action, no recorded schedule."""
    fx, g = load_golden(name)
    rm = backend.RailMap(fx)
    n_dec, n_tick, n_ep = len(g["dec_action"]), len(g["tick_ep"]), int(g["n_episodes"])
    q_cap = 1 << max(6, int(np.ceil(np.log2(len(g["q_keys"]) * 2 + 16))))
    kw = {} if lanes is None else dict(lanes=lanes)
    eng = factory(rm, n_envs=n_envs, q_cap=q_cap, dec_cap=n_dec + 4, tick_cap=n_tick + 4, ep_cap=n_ep + 1, trace_sem=True,
                  rng="reference", malfunction_rng="reference", **kw)
    assert "KIND=full" in eng.kernel_variant(backend.MODE_LEARN)
    eng.set_hparams(**hparams(g), seeds=np.full(n_envs, int(g["seed"])), episodes=n_ep)
    eng.reset()
    eng.enable_q_init(True)
    total = n_tick + 8
    for _ in range(0, total + (chunk or total), chunk or total):
        eng.run(backend.MODE_LEARN, chunk or total)
    c = eng.counters()
    assert (c["err"] == 0).all() and (c["halted"] == 1).all() and (c["decisions"] == n_dec).all(), c
    n, log, delays = eng.episode_log()
    gq = q_dict(g["q_keys"], g["q_vals"])
    exact = float(g["hp_lr_decay_rate"]) == 1.0
    want_state = golden_draws(g)
    want_applied = {tuple(int(x) for x in e) for e in golden_events(g)}
    for env in range(n_envs):
        sched = eng.malfunction_schedule(env)
        got_applied = set()
        for ticks in np.bincount(g["tick_ep"]):
            got_applied |= set(applied_events(sched, rm.trains.T, int(ticks)))
        assert got_applied == want_applied, name
        compare_trace(name, rm, g, *eng.trace(env))
        assert np.array_equal(log[env, :n_ep]["cum_reward"], g["ep_cum_reward"])
        assert np.array_equal(log[env, :n_ep]["arrived"], g["ep_arrived"])
        assert np.array_equal(log[env, :n_ep]["num_malfunctions"], g["ep_num_malfunctions"])
        assert np.array_equal(delays[env, :n_ep].astype(np.float64), g["ep_delays"])
        q = eng.export_q(env, include_init=True)
        assert set(q) == set(gq)
        for k, row in gq.items():
            assert q[k] == row if exact else np.allclose(q[k], row, rtol=1e-12, atol=0.0), k
        assert eng.rng_state(env) == want_state, env
    eng.close()


def test_malfunction_goldens_are_known():
    assert MALF_GOLDENS == ["c1_synth18", "c4_rail100_t50", "c4_synth100_t50", "slips24_t6"]


@pytest.mark.parametrize("name", MALF_GOLDENS)
def test_emul_golden_from_its_seed_alone(name):
    build_emul()
    check_golden_from_seed(name, EmulEngine, chunk=37 if name in ("c1_synth18", "slips24_t6") else None)


# ---------------------------------------------------------------------------------------------- free runs against the oracle
def check_free_run(factory, fx, hp, n_ep, seeds, max_steps=100_000, q_cap=4096, chunk=None, **engine_kw):
    """The oracle free-runs learn() per seed (its own RandomState per episode); the engine free-runs with both streams on
    the device and no bound schedule: every decision, the episode metrics, the Q table, the stream's state and the applied
    malfunctions must agree."""
    rm = backend.RailMap(fx)
    oracles = []
    for sd in seeds:
        try:
            oracles.append((sd, oracle_learn(fx, rm.tab, sd, hp, n_ep, max_steps)))
        except RuntimeError as ex:                 # the reference dies here too (observer.py:294-307)
            if "No train detected" not in str(ex):
                raise
    if not oracles:
        pytest.skip("the reference itself fails on this map for every seed")
    seeds = [sd for sd, _ in oracles]
    n_dec = max(len(o.trace["dec_action"]) for _, o in oracles)
    eng = factory(rm, n_envs=len(seeds), q_cap=q_cap, max_steps=max_steps, dec_cap=n_dec + 4, ep_cap=n_ep + 2,
                  rng="reference", malfunction_rng="reference", **engine_kw)
    eng.set_hparams(**hp, seeds=np.asarray(seeds), episodes=n_ep)
    eng.reset()
    eng.enable_q_init(True)
    for _ in range(1 if chunk is None else 100_000 // chunk):
        eng.run(backend.MODE_LEARN, 1_000_000 if chunk is None else chunk)
        if (eng.counters()["halted"] == 1).all():
            break
    eng.check_errors()
    assert (eng.counters()["halted"] == 1).all()
    _, log, delays = eng.episode_log()
    malfunctions = 0
    for i, (sd, o) in enumerate(oracles):
        dec, _, _ = eng.trace(i)
        t = o.trace
        assert len(dec) == len(t["dec_action"]), (sd, len(dec), len(t["dec_action"]))
        for k_mine, k_o in (("sw", "dec_switch"), ("train", "dec_train"), ("action", "dec_action"), ("next_sw", "dec_next_switch"),
                            ("tick", "dec_tick"), ("done", "dec_done")):
            assert np.array_equal(dec[k_mine], np.array(t[k_o])), (sd, k_mine)
        assert [int(a) | (int(b) << 64) for a, b in zip(dec["arrived"], dec["arrived_hi"])] == [int(x) for x in t["dec_arrived"]], sd
        assert np.array_equal(dec["reward"].astype(np.float64), np.array(t["dec_reward"])), sd
        sched = eng.malfunction_schedule(i)
        applied = set()
        for e_i, ep in enumerate(o.eps):
            assert log[i, e_i]["cum_reward"] == ep["cum_reward"] and log[i, e_i]["decisions"] == ep["decisions"], (sd, e_i)
            assert log[i, e_i]["ticks"] == ep["ticks"] and log[i, e_i]["num_malfunctions"] == ep["num_malfunctions"], (sd, e_i)
            assert list(delays[i, e_i]) == [int(x) for x in ep["delays"]], (sd, e_i)
            applied |= set(applied_events(sched, rm.trains.T, int(ep["ticks"])))
        assert applied == {tuple(int(x) for x in e) for e in o.malfunction_schedule()}, sd
        malfunctions += len(applied)
        assert eng.export_q(i, include_init=True) == o.q_table, sd
        r = np.random.default_rng(int(sd))
        for greedy in t["dec_greedy"]:
            r.random()
            if not greedy:
                r.integers(0, I32MAX)
        assert eng.rng_state(i) == r.bit_generator.state, sd
    eng.close()
    return malfunctions


FREE = [  # (fixture name, hyper-parameters, episodes, seeds, max_steps)
    ("c1_synth18", dict(HP), 4, (450565, 1, 2 ** 32 - 1, 77, 5), 100_000),
    ("slips24_t6", dict(HP, epsilon=0.9, epsilon_decay_rate=0.999, gamma=0.95, default_q=1.5), 3, (64, 3, 12345), 100_000),
    ("slips24_t6", dict(HP, epsilon=0.7), 3, (5, 6), 60),               # episodes cut short by max_steps
    ("c4_rail100_t50", dict(HP, epsilon=0.3), 2, (7, 450565), 100_000),
]


@pytest.mark.parametrize("case", range(len(FREE)))
def test_emul_free_learn_matches_the_oracle(case):
    build_emul()
    name, hp, n_ep, seeds, max_steps = FREE[case]
    fx, _ = load_golden(name)
    n = check_free_run(EmulEngine, fx, hp, n_ep, seeds, max_steps=max_steps, chunk=29 if case == 0 else None)
    assert n > 0                                        # malfunctions took effect


def check_many_trains(factory, name, lanes=None):
    from tests.test_many_trains import HP as HP_T, SEEDS, oracle_runs
    rm = many_train_map(name)
    runs = oracle_runs(name)
    n_dec = max(n for _, _, n, _ in runs)
    kw = {} if lanes is None else dict(lanes=lanes)
    eng = factory(rm, n_envs=len(runs), q_cap=65536, dec_cap=n_dec + 4, ep_cap=2, rng="reference", malfunction_rng="reference", **kw)
    eng.set_hparams(**HP_T, seeds=list(SEEDS), episodes=1)
    eng.reset()
    eng.enable_q_init(True)
    eng.run(backend.MODE_LEARN, 1_000_000)
    eng.check_errors()
    _, log, _ = eng.episode_log()
    for i, (o, eps, n_learn, q_learn) in enumerate(runs):
        dec = eng.trace(i)[0]
        t = o.trace
        for k_mine, k_o in (("sw", "dec_switch"), ("train", "dec_train"), ("action", "dec_action"), ("next_sw", "dec_next_switch")):
            assert np.array_equal(dec[k_mine], np.array(t[k_o][:n_learn])), (name, lanes, k_mine)
        assert [int(a) | (int(b) << 64) for a, b in zip(dec["arrived"], dec["arrived_hi"])] == [int(x) for x in t["dec_arrived"][:n_learn]]
        assert log[i, 0]["cum_reward"] == eps[0]["cum_reward"] and log[i, 0]["decisions"] == eps[0]["decisions"]
        assert log[i, 0]["num_malfunctions"] == eps[0]["num_malfunctions"]
        assert eng.export_q(i, include_init=True) == q_learn, (name, lanes)
    eng.close()


@pytest.mark.parametrize("name", ("t65", "t100", "t128"))
def test_emul_free_learn_above_64_trains(name):
    build_emul()
    check_many_trains(EmulEngine, name)


# ---------------------------------------------------------------------------------------------- test(), Philox epsilon, AEC, CLI
def check_learn_then_test(env_cls, **kw):
    """The drop-in learn(exploit_freq) then test(): every learning episode, every exploit rollout and the final greedy
    rollout are the oracle's, malfunctions included."""
    from oracle.switchfl_oracle import SwitchFLOracle
    fx, _ = load_golden("slips24_t6")
    env = env_cls(api.RailEnv(fx), max_steps=100_000, n_envs=3, q_cap=1024, ep_cap=4, rng="reference", malfunction_rng="reference", **kw)
    hp = dict(HP, epsilon=0.6, epsilon_decay_rate=0.999)
    model = api.DistrQLearning(env=env, seed=64, **hp)
    oracles = [SwitchFLOracle(fx, env.rail_map.tab, seed=64 + i, **hp) for i in range(3)]
    model.learn(num_episodes=5, out_dir=None, checkpoint_freq=0, exploit_freq=2)
    cum, arrived, delays = model.test(out_dir=None, plot=False, save_outputs=False, _batched=True)
    malf = 0
    for i, o in enumerate(oracles):
        eps, exploit = oracle_learn_call(o, 64 + i, 5, exploit_freq=2)
        assert list(model.metrics["cum_reward"][i]) == [e["cum_reward"] for e in eps], i
        assert list(model.metrics["num_malfunctions"][i]) == [e["num_malfunctions"] for e in eps], i
        assert list(model.metrics["cum_reward_exploit"][:, i]) == [e["cum_reward"] for e in exploit], i
        t = o.test()
        assert cum[i] == t["cum_reward"] and arrived[i] == t["arrived"] and list(delays[i]) == [float(x) for x in t["delays"]], i
        assert env.engine.export_q(i, include_init=True) == o.q_table, i
        malf += sum(e["num_malfunctions"] for e in eps) + t["num_malfunctions"]
    assert malf > 0


def test_emul_learn_then_test_matches_the_oracle():
    build_emul()
    check_learn_then_test(EmulSwitchEnv)


def check_philox_epsilon(factory, **kw):
    """rng="philox" with malfunction_rng="reference": the decisions are Philox's, the malfunctions flatland's -- every
    tick's malfunction counters are the schedule's, filtered by the counter rule."""
    fx, _ = load_golden("slips24_t6")
    rm = backend.RailMap(fx)
    seeds = [64, 3, 12345, 0]
    eng = factory(rm, n_envs=len(seeds), q_cap=4096, tick_cap=4 * int(fx["max_episode_steps"]) + 8, ep_cap=5,
                  malfunction_rng="reference", **kw)
    assert "KIND=full" in eng.kernel_variant(backend.MODE_LEARN)
    eng.set_hparams(**HP, seeds=seeds, episodes=4)
    eng.reset()
    eng.enable_q_init(True)
    eng.run(backend.MODE_LEARN, 1_000_000)
    eng.check_errors()
    _, log, _ = eng.episode_log()
    T = rm.trains.T
    total = 0
    for i in range(len(seeds)):
        sched = eng.malfunction_schedule(i)
        tick = eng.trace(i)[1]
        k = 0
        for e_i in range(4):
            ticks = int(log[i, e_i]["ticks"])
            counter, by_tick = [0] * T, {}
            for tk, t, d in sched:
                by_tick.setdefault(int(tk), []).append((int(t), int(d)))
            for now in range(1, ticks + 1):
                for t, d in by_tick.get(now, []):
                    if counter[t] == 0 and d > 0:
                        counter[t] = d
                        total += 1
                counter = [max(c - 1, 0) for c in counter]
                assert list(tick["malf"][k]) == counter, (i, e_i, now)
                k += 1
        assert k == len(tick)
    assert total > 0
    eng.close()


def test_emul_philox_epsilon_with_flatlands_malfunctions():
    build_emul()
    check_philox_epsilon(EmulEngine)


@pytest.mark.parametrize("name", ("c1_synth18", "slips24_t6"))
def test_emul_aec_protocol_with_flatlands_malfunctions(name):
    """reset(seed=s) / agent_iter / last / step: the golden's observations, rewards and arrivals, malfunctions included,
    with no recorded schedule."""
    from tests.test_emul_parity import check_aec
    build_emul()
    fx, g = load_golden(name)
    env = EmulSwitchEnv(api.RailEnv(fx), max_steps=100_000, n_envs=1, q_cap=64, ep_cap=2, malfunction_rng="reference")
    check_aec(env, g)


def test_emul_cli_and_ini():
    build_emul()
    fx, _ = load_golden("slips24_t6")
    with tempfile.TemporaryDirectory() as out:
        cfg = configparser.ConfigParser()
        cfg["MISC"] = {"random_seed": "64", "out_dir": out, "checkpoint_freq": "0", "exploit_freq": "0", "n_envs": "2",
                       "q_cap": "1024", "rng": "reference", "malfunction_rng": "reference"}
        cfg["ENV"] = {"fixture": os.path.join(ROOT, "tests", "golden", "slips24_t6.fixture.npz"), "width": "24", "height": "24",
                      "number_of_agents": "6", "malfunction_rate": str(float(fx["malfunction_rate"])),
                      "min_duration": str(int(fx["min_duration"])), "max_duration": str(int(fx["max_duration"]))}
        cfg["MODEL"] = {k: str(v) for k, v in HP.items()} | {"num_episodes": "3"}
        path = os.path.join(out, "config.ini")
        with open(path, "w") as f:
            cfg.write(f)
        model = cli.launch_experiment(path, device="cpu", env_cls=EmulSwitchEnv)
        assert model.env.engine.malfunction_rng == "reference"
        o = oracle_learn(fx, model.env.rail_map.tab, 64, HP, 3)
        with np.load(os.path.join(out, "cum_reward.npz")) as z:
            assert list(z["x"]) == [e["cum_reward"] for e in o.eps]
        with np.load(os.path.join(out, "num_malfunctions.npz")) as z:
            assert list(z["x"]) == [e["num_malfunctions"] for e in o.eps] and sum(z["x"]) > 0
        with open(os.path.join(out, "distr_q_model.pkl"), "rb") as f:
            assert {tuple(int(x) for x in k): v for k, v in pickle.load(f).items()} == o.q_table
        cfg["MISC"]["malfunction_rng"] = "philox"            # the command-line flag overrides the INI key
        with open(path, "w") as f:
            cfg.write(f)
        env_seen = []

        class Spy(EmulSwitchEnv):
            def __init__(self, *a, **kw):
                env_seen.append(kw["malfunction_rng"])
                super().__init__(*a, **kw)
        cli.launch_experiment(path, device="cpu", env_cls=Spy, malfunction_rng="reference")
        assert env_seen == ["reference"]
        with pytest.raises(SystemExit):
            cli.main(["-c", path, "--malfunction-rng", "mt"])


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_schedule_matches_numpy_and_refusals():
    check_schedules(gpu_engine)
    check_refusals(gpu_engine)


@pytest.mark.gpu
@pytest.mark.parametrize("name", MALF_GOLDENS)
def test_gpu_golden_from_its_seed_alone_at_every_lane_width(name):
    for lanes in (1, 2, 4, 8, 16, 32):
        check_golden_from_seed(name, gpu_engine, lanes=lanes, chunk=53 if lanes == 4 else None)


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(FREE)))
def test_gpu_free_learn_matches_the_oracle(case):
    name, hp, n_ep, seeds, max_steps = FREE[case]
    fx, _ = load_golden(name)
    for lanes in (1, 2, 4, 8, 16, 32):
        check_free_run(gpu_engine, fx, hp, n_ep, seeds, max_steps=max_steps, lanes=lanes)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ("t65", "t100", "t128"))
def test_gpu_free_learn_above_64_trains_at_every_lane_width(name):
    for lanes in (8, 16, 32):
        check_many_trains(gpu_engine, name, lanes=lanes)


@pytest.mark.gpu
def test_gpu_learn_test_philox_epsilon_and_aec():
    from tests.test_emul_parity import check_aec
    for lanes in (1, 2, 4, 8, 16, 32):
        check_learn_then_test(api.ASyncSwitchEnv, _engine_kwargs={"lanes": lanes})
        check_philox_epsilon(gpu_engine, lanes=lanes)
    for name in ("c1_synth18", "slips24_t6"):
        fx, g = load_golden(name)
        env = api.ASyncSwitchEnv(api.RailEnv(fx), max_steps=100_000, n_envs=1, q_cap=64, ep_cap=2, malfunction_rng="reference")
        check_aec(env, g)
