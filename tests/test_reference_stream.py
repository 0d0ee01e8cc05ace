"""The reference's epsilon-greedy stream on the device (``Engine(rng="reference")``, SFL_RNG_REFERENCE).

The reference learner draws from numpy: ``rng = np.random.default_rng(seed)`` per learn() (distr_q.py:269), ``rng.random()``
per decision and, when it explores, ``Generator(PCG64(SeedSequence(rng.integers(0, 2**31 - 1)))).choice(allowed)``
(:315-317).  With that stream on the device a seeded learn() is checked against the reference without recorded actions:
every golden is reproduced from its seed alone (plus its malfunction schedule), and free-running learn() against the oracle,
whose learn() draws from numpy exactly like the reference.  CPU tests run the host build of the device sources (tests/emul);
``-m gpu`` the CUDA kernels at every lane width."""
import configparser
import ctypes as C
import functools
import os
import pickle
import tempfile

import numpy as np
import pytest

from switchfl_b200 import api, backend, cli
from tests._parity import compare_trace, golden_events
from tests._util import golden_names, hparams, load_golden, q_dict
from tests.emulated import EmulEngine, EmulSwitchEnv, build_emul, emul_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
I32MAX = 2 ** 31 - 1
EXPLORE = 1 << 63
HP = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)


@pytest.fixture(scope="module")
def lib():
    return emul_library()


def gpu_engine(*a, **kw):
    return backend.Engine(*a, **kw)


def words(state: dict):
    s, i = state["state"]["state"], state["state"]["inc"]
    return [s >> 64, s & (2 ** 64 - 1), i >> 64, i & (2 ** 64 - 1), state["has_uint32"], state["uinteger"]]


def special_seeds(n_random=2000):
    r = np.random.default_rng(1234)
    fixed = [0, 1, 2, 7, 64, 65, 450565, I32MAX, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 40, 2 ** 63, 2 ** 64 - 1]
    return fixed + [int(x) for x in r.integers(0, 2 ** 63, n_random // 2)] + [int(x) for x in r.integers(0, 2 ** 32, n_random // 2)]


# ---------------------------------------------------------------------------------------------- known answers vs numpy
def check_streams(lib, seeds):
    codes = [0, I32MAX, 0, 0, I32MAX, I32MAX, 0, 5, 2 ** 32, 1, 0, 3 * 2 ** 30, I32MAX, 0]
    init, res, fin = backend.device_pcg64([[0, s, 0, 0, 0, 0] for s in seeds], [codes] * len(seeds), lib=lib)
    for i, s in enumerate(seeds):
        r = np.random.default_rng(s)
        assert backend.pcg64_state(init[i]) == r.bit_generator.state, s
        for k, c in enumerate(codes):
            want = r.random() if c == 0 else int(r.integers(0, c))
            got = res[i, k].view(np.float64) if c == 0 else int(res[i, k])
            assert got == want, (s, k, c, got, want)
        assert backend.pcg64_state(fin[i]) == r.bit_generator.state, s          # carried half-word included


def check_explore_choice(lib, seeds):
    masks = [(1 << k) - 1 for k in range(1, 10)] + [0b100, 0b1010, 0b100100101, 0b110000001]
    init, res, fin = backend.device_pcg64([[0, s, 0, 0, 0, 0] for s in seeds], [[EXPLORE | m for m in masks]] * len(seeds), lib=lib)
    for i, s in enumerate(seeds):
        r = np.random.default_rng(s)
        for k, m in enumerate(masks):
            sd = int(r.integers(0, I32MAX))
            g = np.random.Generator(np.random.PCG64(np.random.SeedSequence(sd)))
            valid = np.array([a for a in range(16) if (m >> a) & 1])
            assert int(res[i, k]) == int(g.choice(valid)), (s, m)
        assert backend.pcg64_state(fin[i]) == r.bit_generator.state


def check_lemire(lib):
    """Ranges where Lemire's rejection is common, from set states (random and carried half-words)."""
    r = np.random.default_rng(99)
    states = []
    for _ in range(300):
        bg = np.random.PCG64(int(r.integers(0, 2 ** 62)))
        bg.advance(int(r.integers(0, 1000)))
        st = bg.state
        st["has_uint32"], st["uinteger"] = int(r.integers(0, 2)), int(r.integers(0, 2 ** 32))
        states.append(st)
    ranges = [3 * 2 ** 30, 3 * 2 ** 30 + 1, 2 ** 31 + 1, 2 ** 32 - 1, 2 ** 32 - 3, 0xAAAAAAAB]
    codes = [ranges[k % len(ranges)] for k in range(40)]
    _, res, fin = backend.device_pcg64([words(s) for s in states], [codes] * len(states), lib=lib)
    rejected = 0
    for i, st in enumerate(states):
        bg = np.random.PCG64()
        bg.state = st
        gen = np.random.Generator(bg)
        for k, c in enumerate(codes):
            before = bg.state
            assert int(res[i, k]) == int(gen.integers(0, c)), (i, k, c)
            # a draw that consumed more than one 32-bit word was rejected at least once
            rejected += (bg.state["state"]["state"] != before["state"]["state"]) and before["has_uint32"] == 0 and bg.state["has_uint32"] == 0
        assert backend.pcg64_state(fin[i]) == bg.state
    assert rejected > 50, rejected


def correctly_rounded_pow(decay: float, n: int) -> float:
    from decimal import Decimal, localcontext
    with localcontext() as ctx:
        ctx.prec = 60
        return 1.0 if n == 0 else float(Decimal(decay) ** n)


def check_eps_slow_path(lib, n_max=10 ** 7):
    """u < epsilon * decay ** n for draws on both sides of the threshold, though the kernel's running product differs from
    decay ** n.  The kernel's power is correctly rounded; Python's ``decay ** n`` is libm's pow, which may be one ulp off
    (glibc: below 0.52 ulp) -- on such an n the two thresholds are adjacent doubles and only a draw equal to the lower one
    could be decided differently.  Everywhere else the kernel's verdict is Python's."""
    rows, want, python = [], [], []
    differs = 0
    r = np.random.default_rng(5)
    for eps0, decay in ((0.5, 0.9997), (0.4, 0.999), (0.9, 0.99999), (0.5, 1.0), (0.5, 0.0)):
        picks = set(range(2000)) | set(int(x) for x in r.integers(0, n_max, 1500)) | {n_max}
        prod = 1.0
        for n in range(n_max + 1):
            if n in picks:
                ref = eps0 * decay ** n
                exact = eps0 * correctly_rounded_pow(decay, n)
                differs += (eps0 * prod) != ref
                for u in (ref, np.nextafter(ref, 0.0), np.nextafter(ref, 1.0), eps0 * prod, exact, np.nextafter(exact, 0.0)):
                    rows.append([u, eps0, decay, n, prod])
                    want.append(u < exact)
                    python.append(u < ref)
            prod *= decay
            if decay in (0.0, 1.0) and n > 2000:
                break
    got = backend.device_explore(rows, lib=lib)
    want, python = np.array(want), np.array(python)
    assert differs > 100, differs                       # the running product is off: the slow path is needed, and taken
    assert np.array_equal(got, want), np.nonzero(got != want)[0][:10]
    assert (got != python).mean() < 1e-3, (got != python).sum()


def test_stream_matches_numpy(lib):
    check_streams(lib, special_seeds())


def test_exploration_matches_numpy_choice(lib):
    check_explore_choice(lib, special_seeds(400))


def test_lemire_rejection_matches_numpy(lib):
    check_lemire(lib)


def test_epsilon_comparison_is_the_references(lib):
    check_eps_slow_path(lib)


# ---------------------------------------------------------------------------------------------- goldens from the seed alone
def golden_draws(g):
    """The reference's generator after a golden's learn(): random() per decision, integers() where it explored."""
    r = np.random.default_rng(int(g["seed"]))
    for greedy in g["dec_greedy"]:
        r.random()
        if not greedy:
            r.integers(0, I32MAX)
    return r.bit_generator.state


def check_golden_free_run(name, factory, n_envs=2, lanes=None, chunk=None):
    fx, g = load_golden(name)
    rm = backend.RailMap(fx)
    n_dec, n_tick, n_ep = len(g["dec_action"]), len(g["tick_ep"]), int(g["n_episodes"])
    ev = golden_events(g)
    q_cap = 1 << max(6, int(np.ceil(np.log2(len(g["q_keys"]) * 2 + 16))))
    kw = {} if lanes is None else dict(lanes=lanes)
    eng = factory(rm, n_envs=n_envs, q_cap=q_cap, dec_cap=n_dec + 4, tick_cap=n_tick + 4, ep_cap=n_ep + 1, ev_cap=len(ev) + 2,
                  trace_sem=True, rng="reference", **kw)
    assert "KIND=full" in eng.kernel_variant(backend.MODE_LEARN)
    eng.set_hparams(**hparams(g), seeds=np.full(n_envs, int(g["seed"])), episodes=n_ep)
    eng.set_replay(None, [ev] * n_envs)                # the malfunction schedule only: no recorded action
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
    for env in range(n_envs):
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


@pytest.mark.parametrize("name", golden_names())
def test_emul_golden_from_its_seed(name):
    build_emul()
    check_golden_free_run(name, EmulEngine, chunk=37 if name.startswith("c1") else None)


# ---------------------------------------------------------------------------------------------- seeds beyond the goldens
def oracle_learn(fx, tab, seed, hp, n_ep, max_steps=100_000):
    from oracle.switchfl_oracle import SwitchFLOracle
    o = SwitchFLOracle(fx, tab, seed=int(seed), max_steps=max_steps, **hp)
    o.enable_trace()
    o.eps = o.learn(n_ep)
    return o


def check_oracle_free_run(factory, fx, hp, n_ep, seeds, max_steps=100_000, q_cap=4096, chunk=None, **engine_kw):
    """The oracle free-runs learn() per seed; the engine free-runs too, on the reference's stream, with the oracle's
    malfunction schedule bound: every decision, the episode metrics, the Q table and the stream's state must agree."""
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
    evs = [o.malfunction_schedule() for _, o in oracles]
    n_dec = max(len(o.trace["dec_action"]) for _, o in oracles)
    eng = factory(rm, n_envs=len(seeds), q_cap=q_cap, max_steps=max_steps, dec_cap=n_dec + 4, ev_cap=max(len(e) for e in evs) + 2,
                  ep_cap=n_ep + 2, rng="reference", **engine_kw)
    eng.set_hparams(**hp, seeds=np.asarray(seeds), episodes=n_ep)
    eng.set_replay(None, evs)
    eng.reset()
    eng.enable_q_init(True)
    for _ in range(1 if chunk is None else 100_000 // chunk):
        eng.run(backend.MODE_LEARN, 1_000_000 if chunk is None else chunk)
        if (eng.counters()["halted"] == 1).all():
            break
    eng.check_errors()
    assert (eng.counters()["halted"] == 1).all()
    _, log, delays = eng.episode_log()
    for i, (sd, o) in enumerate(oracles):
        dec, _, _ = eng.trace(i)
        t = o.trace
        assert len(dec) == len(t["dec_action"]), (sd, len(dec), len(t["dec_action"]))
        for k_mine, k_o in (("sw", "dec_switch"), ("train", "dec_train"), ("action", "dec_action"), ("next_sw", "dec_next_switch"),
                            ("tick", "dec_tick"), ("done", "dec_done")):
            assert np.array_equal(dec[k_mine], np.array(t[k_o])), (sd, k_mine)
        assert [int(a) | (int(b) << 64) for a, b in zip(dec["arrived"], dec["arrived_hi"])] == [int(x) for x in t["dec_arrived"]], sd
        assert np.array_equal(dec["reward"].astype(np.float64), np.array(t["dec_reward"])), sd
        for e_i, ep in enumerate(o.eps):
            assert log[i, e_i]["cum_reward"] == ep["cum_reward"] and log[i, e_i]["decisions"] == ep["decisions"], (sd, e_i)
            assert log[i, e_i]["ticks"] == ep["ticks"] and log[i, e_i]["num_malfunctions"] == ep["num_malfunctions"], (sd, e_i)
            assert list(delays[i, e_i]) == [int(x) for x in ep["delays"]], (sd, e_i)
        assert eng.export_q(i, include_init=True) == o.q_table, sd
        r = np.random.default_rng(int(sd))
        for greedy in t["dec_greedy"]:
            r.random()
            if not greedy:
                r.integers(0, I32MAX)
        assert eng.rng_state(i) == r.bit_generator.state, sd
    eng.close()


FUZZ = [  # (fixture name or mapgen args, hyper-parameters, episodes, seeds, max_steps)
    ("c1_synth18", dict(HP), 4, (450565, 1, 2 ** 32 - 1, 77), 100_000),     # (flatland seeds are 32-bit)
    ("slips24_t6", dict(HP, epsilon=0.9, epsilon_decay_rate=0.999, gamma=0.95, default_q=1.5), 3, (64, 3, 12345), 100_000),
    ("synth40_t12", dict(HP, epsilon=0.3, epsilon_decay_rate=0.99, lr=0.3), 2, (65, 9), 100_000),
    ("loop_chord_7x7", dict(HP, epsilon=1.0, epsilon_decay_rate=1.0), 5, (0, 7, 2 ** 31), 100_000),
    ("slips24_t6", dict(HP, epsilon=0.7), 3, (5, 6), 60),               # episodes cut short by max_steps
]


@pytest.mark.parametrize("case", range(len(FUZZ)))
def test_emul_free_learn_matches_the_oracle(case):
    build_emul()
    name, hp, n_ep, seeds, max_steps = FUZZ[case]
    fx, _ = load_golden(name)
    check_oracle_free_run(EmulEngine, fx, hp, n_ep, seeds, max_steps=max_steps, chunk=29 if case == 0 else None)


@functools.lru_cache(maxsize=None)
def many_train_map(name):
    from tests.test_many_trains import rail_map
    return rail_map(name)


@pytest.mark.parametrize("name", ("t65", "t100", "t128"))
def test_emul_free_learn_above_64_trains(name):
    build_emul()
    from tests.test_many_trains import HP as HP_T, SEEDS, oracle_runs
    rm = many_train_map(name)
    for (o, eps, n_learn, q_learn), sd in zip(oracle_runs(name), SEEDS):
        eng = EmulEngine(rm, n_envs=1, q_cap=65536, dec_cap=n_learn + 4, ev_cap=len(o.malfunction_schedule()) + 2, ep_cap=2, rng="reference")
        eng.set_hparams(**HP_T, seeds=[sd], episodes=1)
        eng.set_replay(None, [o.malfunction_schedule()])
        eng.reset()
        eng.enable_q_init(True)
        eng.run(backend.MODE_LEARN, 1_000_000)
        eng.check_errors()
        dec = eng.trace(0)[0]
        t = o.trace
        for k_mine, k_o in (("sw", "dec_switch"), ("train", "dec_train"), ("action", "dec_action"), ("next_sw", "dec_next_switch")):
            assert np.array_equal(dec[k_mine], np.array(t[k_o][:n_learn])), (name, sd, k_mine)
        assert [int(a) | (int(b) << 64) for a, b in zip(dec["arrived"], dec["arrived_hi"])] == [int(x) for x in t["dec_arrived"][:n_learn]]
        _, log, _ = eng.episode_log()
        assert log[0, 0]["cum_reward"] == eps[0]["cum_reward"] and log[0, 0]["decisions"] == eps[0]["decisions"]
        assert eng.export_q(0, include_init=True) == q_learn, (name, sd)
        eng.close()


# ---------------------------------------------------------------------------------------------- API and CLI
def no_malf(fx):
    fx = dict(fx)
    fx["malfunction_rate"] = 0.0
    return fx


def oracle_learn_call(o, rng_seed, n_ep, exploit_freq=None):
    """distr_q.py:244-379 as the drop-in learn() schedules it: test() before episode t when (t + 1) % exploit_freq == 0."""
    rng = np.random.default_rng(rng_seed)
    o.agent_num_interactions = [0] * o.S                # per learn() call (:263)
    o._q_inited = False                                 # __init_q_table at the first episode of every learn() (:299-300)
    eps, exploit = [], []
    for t in range(n_ep):
        if exploit_freq and (t + 1) % exploit_freq == 0:
            exploit.append(o.test())
        o.episode = t
        eps.append(o.run_episode(rng, greedy=False, learn=True))
    return eps, exploit


def test_emul_api_learn_makes_the_oracles_decisions():
    """ASyncSwitchEnv(rng="reference") + learn(exploit_freq, checkpoint_freq): env i learns on seed + i and writes the
    oracle's curves and Q table; a second learn() restarts the stream."""
    from oracle.switchfl_oracle import SwitchFLOracle
    build_emul()
    fx, _ = load_golden("c1_synth18")
    fx = no_malf(fx)
    env = EmulSwitchEnv(api.RailEnv(fx), max_steps=100_000, n_envs=3, q_cap=1024, ep_cap=4, rng="reference")
    hp = dict(HP, epsilon=0.6, epsilon_decay_rate=0.999)
    model = api.DistrQLearning(env=env, seed=450565, **hp)
    oracles = [SwitchFLOracle(fx, env.rail_map.tab, seed=450565 + i, **hp) for i in range(3)]
    with tempfile.TemporaryDirectory() as out:
        for call in range(2):
            model.learn(num_episodes=7, out_dir=out, checkpoint_freq=3, exploit_freq=2)
            model.write_outputs(0, out)
            for i, o in enumerate(oracles):
                eps, exploit = oracle_learn_call(o, 450565 + i, 7, exploit_freq=2)
                assert list(model.metrics["cum_reward"][i]) == [e["cum_reward"] for e in eps], (call, i)
                assert list(model.metrics["arrived_trains"][i]) == [e["arrived"] for e in eps], (call, i)
                assert list(model.metrics["cum_reward_exploit"][:, i]) == [e["cum_reward"] for e in exploit], (call, i)
                assert env.engine.export_q(i, include_init=True) == o.q_table, (call, i)
            with np.load(os.path.join(out, "cum_reward.npz")) as z:
                assert list(z["x"]) == list(model.metrics["cum_reward"][0])
            with open(os.path.join(out, "distr_q_model.pkl"), "rb") as f:
                q = pickle.load(f)
            assert {tuple(int(x) for x in k): v for k, v in q.items()} == oracles[0].q_table


def test_emul_cli_with_the_reference_stream():
    from oracle.switchfl_oracle import SwitchFLOracle
    build_emul()
    with tempfile.TemporaryDirectory() as out:
        cfg = configparser.ConfigParser()
        cfg["MISC"] = {"random_seed": "450565", "out_dir": out, "checkpoint_freq": "0", "exploit_freq": "0", "n_envs": "2",
                       "q_cap": "1024", "rng": "reference"}
        cfg["ENV"] = {"fixture": os.path.join(ROOT, "tests", "golden", "c1_synth18.fixture.npz"), "width": "18", "height": "18",
                      "number_of_agents": "2", "malfunction_rate": "0", "min_duration": "0", "max_duration": "0"}
        cfg["MODEL"] = {k: str(v) for k, v in HP.items()} | {"num_episodes": "5"}
        path = os.path.join(out, "config.ini")
        with open(path, "w") as f:
            cfg.write(f)
        model = cli.launch_experiment(path, device="cpu", env_cls=EmulSwitchEnv)
        assert model.env.engine.rng == "reference"
        fx, _ = load_golden("c1_synth18")
        o = oracle_learn(no_malf(fx), model.env.rail_map.tab, 450565, HP, 5)
        with np.load(os.path.join(out, "cum_reward.npz")) as z:
            assert list(z["x"]) == [e["cum_reward"] for e in o.eps]
        with open(os.path.join(out, "distr_q_model.pkl"), "rb") as f:
            assert {tuple(int(x) for x in k): v for k, v in pickle.load(f).items()} == o.q_table


def test_refusals_are_loud(lib):
    build_emul()
    fx, _ = load_golden("c1_synth18")
    rm = backend.RailMap(fx)
    with pytest.raises(RuntimeError, match="shared-table"):
        EmulEngine(rm, n_envs=2, q_cap=2, shared_q=True, rng="reference")
    with pytest.raises(ValueError, match="rng must be one of"):
        EmulEngine(rm, n_envs=2, rng="pcg")
    cfg = backend.Config(n_envs=2, q_cap=1024, pend_cap=8, max_steps=100, ep_cap=1, rng=2)
    assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(backend.Sizes())) == -1
    assert b"rng must be" in lib.sfl_last_error()
    old = backend.ABI_VERSION
    try:
        backend.ABI_VERSION = 7                          # a binding of the previous ABI refuses this library
        with pytest.raises(RuntimeError, match="ABI version mismatch"):
            backend.load_library(build_emul())
    finally:
        backend.ABI_VERSION = old
    eng = EmulEngine(rm, n_envs=1)
    with pytest.raises(RuntimeError, match="rng_state"):
        eng.rng_state()


@pytest.mark.parametrize("name", ("c1_synth18", "c4_rail100_t50"))
def test_sizes_unchanged_without_the_reference_stream(lib, name):
    fx, _ = load_golden(name)
    rm = backend.RailMap(fx)
    sizes = {}
    for rng in (0, 1):
        cfg = backend.Config(n_envs=16, q_cap=1024, pend_cap=8, max_steps=100, dec_cap=4, ep_cap=2, rng=rng)
        s = backend.Sizes()
        assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(s)) == 0
        sizes[rng] = {k: getattr(s, k) for k, _ in backend.Sizes._fields_}
    assert sizes[0]["rng_offset"] == 0 and sizes[1]["rng_offset"] == 248 + (32 if rm.trains.T > 64 else 0)
    # the 48-byte block fits in the header's alignment padding or adds to the stride; nothing else moves
    assert {k: v for k, v in sizes[0].items() if k not in ("rng_offset", "env_stride", "state_bytes")} == \
           {k: v for k, v in sizes[1].items() if k not in ("rng_offset", "env_stride", "state_bytes")}
    cfg = backend.Config(n_envs=16, q_cap=1024, pend_cap=8, max_steps=100, dec_cap=4, ep_cap=2)     # zero-initialised: Philox
    s = backend.Sizes()
    assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(s)) == 0
    assert {k: getattr(s, k) for k, _ in backend.Sizes._fields_} == sizes[0]


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_known_answers():
    lib = backend.load_library()
    check_streams(lib, special_seeds())
    check_explore_choice(lib, special_seeds(400))
    check_lemire(lib)
    check_eps_slow_path(lib)


@pytest.mark.gpu
@pytest.mark.parametrize("name", golden_names())
def test_gpu_golden_from_its_seed_at_every_lane_width(name):
    for lanes in (1, 2, 4, 8, 16, 32):
        check_golden_free_run(name, gpu_engine, lanes=lanes, chunk=53 if lanes == 4 else None)


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(FUZZ)))
def test_gpu_free_learn_matches_the_oracle(case):
    name, hp, n_ep, seeds, max_steps = FUZZ[case]
    fx, _ = load_golden(name)
    for lanes in (1, 8, 32):
        check_oracle_free_run(gpu_engine, fx, hp, n_ep, seeds, max_steps=max_steps, lanes=lanes)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ("t65", "t100", "t128"))
def test_gpu_free_learn_above_64_trains_at_every_lane_width(name):
    from tests.test_many_trains import HP as HP_T, SEEDS, oracle_runs
    rm = many_train_map(name)
    runs = oracle_runs(name)
    evs = [o.malfunction_schedule() for o, _, _, _ in runs]
    n_dec = max(n for _, _, n, _ in runs)
    for lanes in (8, 16, 32):
        eng = backend.Engine(rm, n_envs=len(runs), q_cap=65536, dec_cap=n_dec + 4, ev_cap=max(len(e) for e in evs) + 2, ep_cap=2,
                             rng="reference", lanes=lanes)
        assert eng.kernel_variant(backend.MODE_LEARN).endswith(",NW=2>") and "KIND=full" in eng.kernel_variant(backend.MODE_LEARN)
        eng.set_hparams(**HP_T, seeds=list(SEEDS), episodes=1)
        eng.set_replay(None, evs)
        eng.reset()
        eng.enable_q_init(True)
        eng.run(backend.MODE_LEARN, 1_000_000)
        eng.check_errors()
        for i, (o, eps, n_learn, q_learn) in enumerate(runs):
            dec = eng.trace(i)[0]
            for k_mine, k_o in (("sw", "dec_switch"), ("train", "dec_train"), ("action", "dec_action"), ("next_sw", "dec_next_switch")):
                assert np.array_equal(dec[k_mine], np.array(o.trace[k_o][:n_learn])), (name, lanes, k_mine)
            assert eng.export_q(i, include_init=True) == q_learn, (name, lanes)
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ("c4", "t100"))
def test_gpu_properties_at_the_benchmark_batch(which):
    """scripts/bench_ref_stream.py's workloads: no errors, halted, environments with equal seeds identical, and the
    launch it times is the full kernel."""
    from switchfl_b200 import mapgen
    fx, n = (mapgen.c4_fixture(), 8192) if which == "c4" else (mapgen.t100_fixture(), 3552)
    rm = backend.RailMap(fx)
    eng = backend.Engine(rm, n_envs=n, q_cap=16384 if which == "c4" else 65536, ep_cap=4, rng="reference")
    variant = eng.kernel_variant(backend.MODE_LEARN)
    assert variant == "k_run<G=32,KIND=full,TH=0,SQ=0,ONE=0,ROOMY=0" + ("" if which == "c4" else ",NW=2") + ">", variant
    seeds = np.arange(n) // 2 + 450565                  # pairs of environments with equal seeds
    eng.set_hparams(**HP, seeds=seeds, episodes=1)
    eng.reset()
    eng.enable_q_init(True)
    for _ in range(8):
        eng.run(backend.MODE_LEARN, 512)
        if (eng.counters()["halted"] == 1).all():
            break
    eng.check_errors()
    c = eng.counters()
    assert (c["halted"] == 1).all()
    for k in ("decisions", "ticks", "q_rows", "stop_actions", "arrived_trains"):
        assert np.array_equal(c[k][0::2], c[k][1::2]), k
    st = eng.rng_state()
    assert all(st[2 * i] == st[2 * i + 1] for i in range(0, n // 2, 97))
    eng.close()
