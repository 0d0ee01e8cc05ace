"""Maps with more than 64 trains: the train sets take two 64-bit words (the NW = 2 kernels).

Three maps: T = 65 (train 64, the first train of word 1), T = 100 (``mapgen.t100_fixture``, the reference's 100-train
evaluation on the C4 rail network) and T = 128 (both words full, semaphore-holder index 127).  No reference golden exists
above 50 trains; the oracle (pinned by the goldens, no train-count-dependent logic) free-runs and its trace -- recorded in
the golden layout -- is the expected result.  ``tests._parity.check_against_oracle`` checks ``popcount(arrived_mask) ==
arrived``, which only holds for word 0, so the two-word comparisons live here.  CPU tests run the host build of the device
sources (tests/emul); ``-m gpu`` the CUDA kernels."""
import functools
import os
import subprocess
import tempfile

import numpy as np
import pytest

from switchfl_b200 import api, backend, mapgen
from tests.emulated import EmulEngine, EmulSwitchEnv, build_emul

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HP = dict(gamma=0.9, epsilon=0.5, epsilon_decay_rate=0.999, lr=0.2, lr_decay_rate=1.0, default_q=0.5)
SEEDS = (450565, 17)
MAPS = ("t65", "t100", "t128")
WIDE_LANES = (8, 16, 32)


def _make(name):
    if name == "t65":
        return mapgen.rail_fixture(60, 65, 1, n_rings=2, n_lines=10, cross_every=8, num_cities=12, malfunction_rate=0.02,
                                   min_duration=3, max_duration=9, name="rail60_t65")
    if name == "t100":
        return mapgen.t100_fixture()
    if name == "t128":
        return mapgen.rail_fixture(120, 128, 0, n_rings=3, n_lines=24, cross_every=8, num_cities=25, malfunction_rate=0.01,
                                   min_duration=5, max_duration=15, name="rail120_t128")
    raise KeyError(name)


@functools.lru_cache(maxsize=None)
def rail_map(name) -> backend.RailMap:
    return backend.RailMap(_make(name))


@functools.lru_cache(maxsize=None)
def oracle_runs(name):
    """Per seed: the oracle after one free learn() episode and one greedy test() rollout (traced), its episode metrics, the
    number of learn() decisions and the Q table learn() left."""
    from oracle.switchfl_oracle import SwitchFLOracle
    rm = rail_map(name)
    out = []
    for sd in SEEDS:
        o = SwitchFLOracle(rm.fixture, rm.tab, seed=sd, **HP)
        o.enable_trace()
        eps = o.learn(1)
        n_learn = len(o.trace["dec_action"])
        q_learn = {k: list(v) for k, v in o.q_table.items()}
        o.episode = 1
        eps.append(o.test())
        out.append((o, eps, n_learn, q_learn))
    return out


def wide_set(lo, hi) -> int:
    return int(lo) | (int(hi) << 64)


def check_wide_replay(factory, name, **engine_kw):
    """Replay of the oracle's free learn() episode, then a greedy rollout: every decision (switch, train, action, next switch,
    reward, done, the whole arrived set), the episode logs and the Q tables."""
    rm, runs = rail_map(name), oracle_runs(name)
    n_dec = max(len(o.trace["dec_action"]) for o, _, _, _ in runs)
    evs = [o.malfunction_schedule() for o, _, _, _ in runs]
    eng = factory(rm, n_envs=len(runs), q_cap=65536, dec_cap=n_dec + 4, act_cap=n_dec + 4, ev_cap=max(len(e) for e in evs) + 2,
                  ep_cap=3, **engine_kw)
    seeds = np.array(SEEDS)
    eng.set_hparams(**HP, seeds=seeds, episodes=1)
    eng.set_replay([o.replay_stream(0, n) for o, _, n, _ in runs], evs)
    eng.reset()
    eng.enable_q_init(True)
    eng.run(backend.MODE_REPLAY, 1_000_000)
    eng.check_errors()
    assert (eng.counters()["halted"] == 1).all()
    learn_dec = [eng.trace(i)[0].copy() for i in range(len(runs))]
    _, llog, ldelays = eng.episode_log()
    eng.set_hparams(**HP, seeds=seeds, episodes=1, episode_base=1)
    eng.reset(keep_q=True, keep_interactions=True)
    eng.run(backend.MODE_GREEDY, 1_000_000)
    eng.check_errors()
    _, glog, gdelays = eng.episode_log()
    high = 0
    for i, (o, eps, n_learn, _) in enumerate(runs):
        t = o.trace
        greedy_dec = eng.trace(i)[0]
        for dec, first, last in ((learn_dec[i], 0, n_learn), (greedy_dec, n_learn, None)):
            assert len(dec) == len(t["dec_action"][first:last]), (name, i, len(dec))
            for k_mine, k_o in (("sw", "dec_switch"), ("train", "dec_train"), ("action", "dec_action"), ("next_sw", "dec_next_switch"),
                                ("tick", "dec_tick"), ("done", "dec_done")):
                assert np.array_equal(dec[k_mine], np.array(t[k_o][first:last])), (name, i, k_mine)
            assert np.array_equal(dec["reward"].astype(np.float64), np.array(t["dec_reward"][first:last])), (name, i)
            got = [wide_set(a, b) for a, b in zip(dec["arrived"], dec["arrived_hi"])]
            assert got == [int(x) for x in t["dec_arrived"][first:last]], (name, i, "arrived")
            high |= max(got) >> 64
        for rec, delays, ep in ((llog[i, 0], ldelays[i, 0], eps[0]), (glog[i, 0], gdelays[i, 0], eps[1])):
            assert rec["cum_reward"] == ep["cum_reward"] and rec["decisions"] == ep["decisions"] and rec["ticks"] == ep["ticks"], (name, i)
            assert rec["arrived"] == ep["arrived"] == bin(wide_set(rec["arrived_mask"], rec["arrived_mask_hi"])).count("1"), (name, i)
            assert rec["num_malfunctions"] == ep["num_malfunctions"], (name, i)
            assert list(delays) == [int(x) for x in ep["delays"]], (name, i)
        assert eng.export_q(i, include_init=True) == o.q_table, (name, i)
    assert high, "no train of word 1 arrived: the second word went untested"
    eng.close()


# ---------------------------------------------------------------------------------------------- CPU (host build)
@pytest.fixture(scope="module")
def emul_lib():
    return build_emul()


@pytest.mark.parametrize("name", MAPS)
def test_emul_replays_the_oracle_above_64_trains(name, emul_lib):
    check_wide_replay(EmulEngine, name)


def test_emul_aec_protocol_with_100_trains(emul_lib):
    """reset / agent_iter / last / step through the drop-in env on rail100_t100: observations, masks, last() rewards (trains
    of word 1 included), next switches and arrived_trains lists are the oracle's, and a host-side learner on top ends with
    the oracle's Q table."""
    from tests.test_emul_parity import check_aec
    rm = rail_map("t100")
    o, eps, n_learn, q_learn = oracle_runs("t100")[0]
    t = o.trace
    assert max(t["dec_train"][:n_learn]) >= 64
    keys = np.full((len(q_learn), 18), -9, np.int64)
    vals = np.full((len(q_learn), 9), np.nan)
    for r, (k, v) in enumerate(q_learn.items()):
        keys[r, :len(k)] = k
        vals[r, :len(v)] = v
    g = {"hp_" + k: v for k, v in HP.items()}
    g.update(n_episodes=1, seed=SEEDS[0], q_keys=keys, q_vals=vals, ep_cum_reward=[eps[0]["cum_reward"]])
    g.update({k: t[k][:n_learn] for k in ("dec_obs", "dec_mask", "dec_reward", "dec_tick", "dec_switch", "dec_action", "dec_next_switch",
                                           "dec_arrived")})
    ev = o.malfunction_schedule()
    env = EmulSwitchEnv(api.RailEnv(rm.fixture), max_steps=100_000, n_envs=1, q_cap=64, ep_cap=2, _engine_kwargs={"ev_cap": len(ev) + 2})
    env.engine.set_replay(None, [ev])
    check_aec(env, g)
    env.engine.close()


def test_emul_learn_writes_trains_of_word_1(emul_lib, tmp_path):
    """learn() on rail100_t100: trains_at_dest holds the trains 64..99 that arrived, like every other output."""
    env = EmulSwitchEnv(api.RailEnv(rail_map("t100").fixture), max_steps=100_000, n_envs=2, ep_cap=4)
    m = api.DistrQLearning(env=env, **HP, seed=SEEDS[0])
    m.learn(num_episodes=2, out_dir=str(tmp_path), checkpoint_freq=0)
    _, log, _ = env.engine.episode_log()
    for i in range(2):
        want = backend.train_set(log[i, 1]["arrived_mask"], log[i, 1]["arrived_mask_hi"], 100)
        assert m.metrics["trains_at_dest"][i] == want and len(want) == m.metrics["arrived_trains"][i, 1]
    at_dest = np.load(os.path.join(str(tmp_path), "trains_at_dest.npz"))["x"]
    assert list(at_dest) == m.metrics["trains_at_dest"][0] and max(at_dest) >= 64
    assert os.path.exists(os.path.join(str(tmp_path), "delays.npz"))
    env.engine.close()


def test_cli_runs_the_reference_ini_with_100_agents(emul_lib, tmp_path):
    """main.py with the reference's INI schema and number_of_agents = 100 on the synthetic double-track generator: learn()
    runs and writes the reference's output files."""
    import configparser
    from switchfl_b200 import cli
    ini = os.path.join(str(tmp_path), "config.ini")
    out = os.path.join(str(tmp_path), "out")
    c = configparser.ConfigParser()
    c["MISC"] = {"random_seed": 450565, "out_dir": out, "checkpoint_freq": 2, "exploit_freq": 2}
    c["ENV"] = {"width": 100, "height": 100, "max_num_cities": 25, "max_rails_between_cities": 2, "max_rail_pairs_in_city": 2,
                "number_of_agents": 100, "malfunction_rate": 0.01, "min_duration": 5, "max_duration": 15}
    c["MODEL"] = {"gamma": 1.0, "epsilon": 0.5, "epsilon_decay_rate": 0.9997, "lr": 0.1, "lr_decay_rate": 1.0, "default_q": 0.0,
                  "num_episodes": 2}
    with open(ini, "w") as f:
        c.write(f)
    model = cli.launch_experiment(ini, env_cls=EmulSwitchEnv)
    assert model.env.rail_env.get_num_agents() == 100
    for name in ("cum_reward", "arrived_trains", "delays", "num_malfunctions", "trains_at_dest", "cum_reward_exploit",
                 "arrived_trains_exploit", "trains_at_dest_checkpoint_2"):
        assert os.path.exists(os.path.join(out, name + ".npz")), name
    assert os.path.exists(os.path.join(out, "distr_q_model.pkl"))
    assert np.load(os.path.join(out, "delays.npz"))["x"].shape == (2, 100)
    at_dest = np.load(os.path.join(out, "trains_at_dest.npz"))["x"]
    assert len(at_dest) == np.load(os.path.join(out, "arrived_trains.npz"))["x"][-1] and at_dest.max() >= 64
    model.env.engine.close()


def test_more_than_128_trains_fail_loudly(emul_lib):
    fx = mapgen.rail_fixture(120, 129, 0, n_rings=3, n_lines=24, cross_every=8, num_cities=25)
    with pytest.raises(RuntimeError, match=r"1\.\.128"):
        EmulEngine(backend.RailMap(fx), n_envs=1)


def test_shared_table_mode_above_64_trains_fails_loudly(emul_lib):
    with pytest.raises(RuntimeError, match="at most 64 trains"):
        EmulEngine(rail_map("t65"), n_envs=1, q_cap=2, shared_q=True)


def test_fewer_than_8_lanes_above_64_trains_fail_loudly(emul_lib):
    eng = EmulEngine(rail_map("t65"), n_envs=1, bind=False)
    for lanes in (1, 2, 4):
        with pytest.raises(RuntimeError, match="8, 16 or 32 lanes"):
            eng._ck(eng.lib.sfl_set_lanes(eng.ctx, lanes))
    for lanes in WIDE_LANES:
        eng._ck(eng.lib.sfl_set_lanes(eng.ctx, lanes))
    eng.close()


def test_record_fields_for_word_1_sit_where_the_header_puts_them():
    """The appended fields at the offsets the C compiler gives them; the existing fields keep theirs."""
    fields = [("sfl_dec_rec", "arrived"), ("sfl_dec_rec", "arrived_hi"), ("sfl_ep_rec", "arrived_mask"), ("sfl_ep_rec", "arrived_mask_hi"),
              ("sfl_step_rec", "arrived"), ("sfl_step_rec", "rewards"), ("sfl_step_rec", "arrived_hi")]
    prog = "#include <stdio.h>\n#include <stddef.h>\n#include \"switchfl_b200.h\"\nint main(void) {\n" + "".join(
        f'  printf("%zu\\n", offsetof({s}, {f}));\n' for s, f in fields) + "  return 0;\n}\n"
    with tempfile.TemporaryDirectory() as tmp:
        open(os.path.join(tmp, "o.c"), "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(tmp, "o"), os.path.join(tmp, "o.c")])
        got = [int(x) for x in subprocess.check_output([os.path.join(tmp, "o")]).split()]
    dts = {"sfl_dec_rec": backend.DEC_DT, "sfl_ep_rec": backend.EP_DT, "sfl_step_rec": backend.STEP_DT}
    assert got == [dts[s].fields[f][1] for s, f in fields]
    assert got == [40, 48, 24, 32, 32, 40, 552]                      # word 0 and the rewards where ABI 6 had them


# ---------------------------------------------------------------------------------------------- GPU
def gpu_engine(rm, **kw):
    return backend.Engine(rm, device="cuda:0", **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", WIDE_LANES)
@pytest.mark.parametrize("name", MAPS)
def test_cuda_replays_the_oracle_above_64_trains(name, lanes):
    check_wide_replay(gpu_engine, name, lanes=lanes)


def _free_run(cls, rm, lanes, full, B=4, n_ep=2):
    """Free-running learn then one greedy rollout; everything observable, plus the two kernel instantiations."""
    eng = cls(rm, n_envs=B, q_cap=65536, ep_cap=4, lanes=lanes, dec_cap=4 if full else 0)
    kernels = (eng.kernel_variant(backend.MODE_LEARN, traced=full), eng.kernel_variant(backend.MODE_GREEDY, traced=full))
    eng.set_hparams(**HP, seeds=np.arange(B) + 77, episodes=n_ep)
    eng.reset()
    eng.enable_q_init(True)
    eng.run(backend.MODE_LEARN, 1_000_000)
    eng.check_errors()
    c1 = eng.counters().copy()
    _, log1, d1 = eng.episode_log()
    eng.set_hparams(**HP, seeds=np.arange(B) + 77, episodes=1, episode_base=n_ep)
    eng.reset(keep_q=True, keep_interactions=True)
    eng.run(backend.MODE_GREEDY, 1_000_000)
    eng.check_errors()
    c2 = eng.counters().copy()
    _, log2, d2 = eng.episode_log()
    q = [eng.export_q(i) for i in range(B)]
    eng.close()
    return (c1, log1[:, :n_ep].copy(), d1[:, :n_ep].copy(), c2, log2[:, :1].copy(), d2[:, :1].copy(), q), kernels


@functools.lru_cache(maxsize=None)
def _host_free_run(name):
    return _free_run(EmulEngine, rail_map(name), None, False)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", WIDE_LANES)
@pytest.mark.parametrize("name", MAPS)
def test_cuda_wide_production_kernels_equal_the_full_kernel_and_the_host_build(name, lanes):
    """Every NW = 2 instantiation (learn, greedy, full at 8, 16 and 32 lanes): counters, episode logs and Q tables of a free
    run equal those of the full kernel and of the host build."""
    from tests.test_gpu_parity import _assert_same_run
    rm = rail_map(name)
    prod, k_prod = _free_run(gpu_engine, rm, lanes, full=False)
    full, k_full = _free_run(gpu_engine, rm, lanes, full=True)
    assert k_prod == (f"k_run<G={lanes},KIND=learn,TH=0,SQ=0,ONE=0,ROOMY=0,NW=2>", f"k_run<G={lanes},KIND=greedy,TH=0,SQ=0,ONE=0,ROOMY=0,NW=2>")
    assert k_full[0] == f"k_run<G={lanes},KIND=full,TH=0,SQ=0,ONE=0,ROOMY=0,NW=2>", k_full
    _assert_same_run(prod, full)
    _assert_same_run(prod, _host_free_run(name))
    assert (prod[1]["arrived_mask_hi"] != 0).any()


def bench_trains():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_trains", os.path.join(ROOT, "scripts", "bench_trains.py"))
    bt = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bt)
    return bt


@pytest.mark.gpu
def test_cuda_bench_trains_kernel_is_parity_tested():
    """The instantiation scripts/bench_trains.py times is one the test above pins (G = 8, 16 or 32, learn, NW = 2)."""
    bt = bench_trains()
    eng = backend.Engine(rail_map("t100"), n_envs=bt.ENVS, q_cap=bt.Q_CAP, ep_cap=4, bind=False)
    variant = eng.kernel_variant(backend.MODE_LEARN)
    eng.close()
    assert variant in {f"k_run<G={g},KIND=learn,TH=0,SQ=0,ONE=0,ROOMY=0,NW=2>" for g in WIDE_LANES}, variant


@pytest.mark.gpu
def test_cuda_learn_t100_at_the_benchmark_batch_properties():
    """rail100_t100 at the batch scripts/bench_trains.py times: free-running learn; no errors, no abandoned episodes, forced
    stops under 20 %, more than 15 of 100 trains arrive per episode, bookkeeping closes, the same seeds repeat."""
    rm = rail_map("t100")
    B, n_ep, T = bench_trains().ENVS, 2, 100
    eng = gpu_engine(rm, n_envs=B, q_cap=65536, ep_cap=4)
    eng.set_hparams(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0,
                    seeds=np.arange(B) + 450565, episodes=n_ep)
    eng.reset()
    eng.enable_q_init(True)
    eng.run(backend.MODE_LEARN, 100000)
    eng.check_errors()
    c = eng.counters()
    assert (c["halted"] == 1).all() and (c["episodes"] == n_ep).all() and (c["aborted"] == 0).all() and (c["err"] == 0).all()
    assert c["forced_stops"].sum() < 0.2 * c["decisions"].sum() and c["arrived_trains"].sum() > 0.15 * T * n_ep * B
    n, log, _ = eng.episode_log()
    assert (n == n_ep).all()
    assert (log["decisions"][:, :n_ep].sum(axis=1) == c["decisions"]).all()
    assert (log["ticks"][:, :n_ep].sum(axis=1) == c["ticks"]).all()
    assert (log["ticks"][:, :n_ep] <= int(rm.fixture["max_episode_steps"])).all()
    pop = np.array([[bin(wide_set(r["arrived_mask"], r["arrived_mask_hi"])).count("1") for r in row[:n_ep]] for row in log])
    assert (pop == log["arrived"][:, :n_ep]).all()
    assert (log["arrived"][:, :n_ep].sum(axis=1) == c["arrived_trains"]).all()
    d, t = eng.total_decisions()
    assert d == int(c["decisions"].sum()) and t == int(c["ticks"].sum())
    first = c.copy()
    eng.reset()
    eng.run(backend.MODE_LEARN, 100000)
    c2 = eng.counters()
    for k in ("decisions", "ticks", "arrived_trains", "forced_stops"):
        assert np.array_equal(c2[k], first[k]), k
    eng.close()
