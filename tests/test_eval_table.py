"""Evaluation contexts (``Engine(eval_q=True)``, ``DistrQLearning.evaluate``): one read-only Q table, many environments.

The reference evaluates a trained table with ``load()`` + ``test()`` (eval.py:31-97): every evaluation gets a private copy,
and test() inserts a default row at every lookup that misses (distr_q.py:482 -> :56-57).  An evaluation context keeps no
per-environment table; its greedy kernel (k_eval) probes one shared table and inserts nothing.  The expected result is the
existing path: the same table imported into N private tables, then a greedy episode -- per environment the same cumulative
reward, decisions, ticks, arrived trains (both words of the set), malfunctions and delays.  CPU tests run the host build of
the device sources (tests/emul); ``-m gpu`` the CUDA kernels at every lane width of the new instantiations."""
import ctypes as C
import functools
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from switchfl_b200 import api, backend, cli, mapgen
from tests._util import load_golden
from tests.emulated import EmulEngine, EmulSwitchEnv, build_emul

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAPS = ("c1_synth18", "slips24_t6", "c3_rail80_s64", "c4_rail100_t50", "t100")
HP = dict(gamma=0.9, epsilon=0.5, epsilon_decay_rate=0.999, lr=0.2, lr_decay_rate=1.0)
EP_FIELDS = ("cum_reward", "decisions", "ticks", "arrived", "arrived_mask", "arrived_mask_hi", "num_malfunctions")
SEED0 = 1000


@functools.lru_cache(maxsize=None)
def rail_map(name) -> backend.RailMap:
    fx = mapgen.t100_fixture() if name == "t100" else load_golden(name)[0]
    if name == "c3_rail80_s64":                          # the shipped C3 map has none: give it malfunctions
        fx = dict(fx, malfunction_rate=0.02, min_duration=2, max_duration=6)
    return backend.RailMap(fx)


@functools.lru_cache(maxsize=None)
def learned(name, default_q, episodes=2):
    """(the learner's q_table with the optimistic rows, the rows learn() created without them) of a short host-build learn()."""
    rm = rail_map(name)
    env = EmulSwitchEnv(api.RailEnv(rm.fixture), max_steps=100_000, n_envs=1, q_cap=1 << 17)
    m = api.DistrQLearning(env, **HP, default_q=default_q, seed=7)
    m.learn(episodes, None, 0)
    with_init = dict(m.q_table)
    without = env.engine.export_q(0, include_init=False)
    env.engine.close()
    return with_init, without


def table(name, kind, default_q):
    with_init, without = learned(name, default_q)
    if kind == "init":
        return with_init
    if kind == "learned":
        return without
    keys = sorted(with_init)                             # "holes": every third row missing
    return {k: with_init[k] for i, k in enumerate(keys) if i % 3}


def cap_for(q):
    cap = 1024
    while cap < 2 * len(q) + 2:
        cap *= 2
    return cap


def greedy_until_halted(eng):
    for _ in range(1000):
        eng.run(backend.MODE_GREEDY, 512)
        c = eng.counters()
        eng.check_errors()
        if (c["halted"] == 1).all():
            return c
    raise AssertionError("greedy episodes did not end")


def private_run(cls, rm, q, seeds, default_q, **kw):
    """The existing path: load() -- the table into every environment's private table -- then test()."""
    eng = cls(rm, n_envs=len(seeds), q_cap=cap_for(q), ep_cap=1, **kw)
    eng.set_hparams(**HP, default_q=default_q, seeds=seeds, episodes=-1)
    eng.reset()
    for i in range(len(seeds)):
        eng.import_q(i, q)
    eng.set_hparams(**HP, default_q=default_q, seeds=seeds, episodes=1)
    eng.reset(keep_q=True, keep_interactions=True)
    eng.enable_q_init(False)
    c = greedy_until_halted(eng)
    _, log, dl = eng.episode_log()
    eng.close()
    return c, log[:, 0].copy(), dl[:, 0].copy()


def eval_run(cls, rm, q, seeds, default_q, lanes=None, **kw):
    eng = cls(rm, n_envs=len(seeds), q_cap=cap_for(q), ep_cap=1, eval_q=True, lanes=lanes, **kw)
    eng.set_hparams(**HP, default_q=default_q, seeds=seeds, episodes=1)
    eng.reset()
    eng.set_eval_table(q)
    before = eng.buf["eval_q"].cpu().clone()
    c = greedy_until_halted(eng)
    assert np.array_equal(eng.buf["eval_q"].cpu().numpy(), before.numpy()), "the evaluation table was written"
    _, log, dl = eng.episode_log()
    variant = eng.kernel_variant(backend.MODE_GREEDY)
    eng.close()
    return c, log[:, 0].copy(), dl[:, 0].copy(), variant


def assert_same_episodes(got, want, what):
    (gc, glog, gdl), (wc, wlog, wdl) = got[:3], want[:3]
    for f in EP_FIELDS:
        assert np.array_equal(glog[f], wlog[f]), (what, f, glog[f], wlog[f])
    assert np.array_equal(gdl, wdl), (what, "delays")
    assert np.array_equal(gc["decisions"], wc["decisions"]) and np.array_equal(gc["ticks"], wc["ticks"]), what
    assert (gc["q_rows"] == 0).all(), "an evaluation context has no rows of its own"


# ---------------------------------------------------------------------------------------------- CPU (host build)
CASES = [(name, kind, dq) for name in MAPS for kind, dq in (("init", 0.0), ("learned", 0.5), ("holes", 0.5))]


@pytest.mark.parametrize("name,kind,default_q", CASES)
def test_emul_eval_table_equals_private_tables(name, kind, default_q):
    rm = rail_map(name)
    q = table(name, kind, default_q)
    seeds = np.arange(6) + SEED0
    want = private_run(EmulEngine, rm, q, seeds, default_q)
    got = eval_run(EmulEngine, rm, q, seeds, default_q)
    assert_same_episodes(got, want, (name, kind))
    if kind != "init":                                   # lookups missed: test() inserted default rows there
        assert (want[0]["q_rows"] > len(q)).any()
    if rm.trains.T > 64:
        assert (want[1]["arrived_mask_hi"] != 0).any(), "no train of word 1 arrived"
    assert (want[1]["num_malfunctions"] > 0).any(), (name, "no malfunctions: pick another map or seed")


@pytest.mark.parametrize("name", ["slips24_t6", "c4_rail100_t50", "t100"])
def test_emul_eval_table_with_flatland_malfunctions(name):
    rm = rail_map(name)
    q = table(name, "holes", 0.5)
    seeds = np.arange(5) + SEED0
    want = private_run(EmulEngine, rm, q, seeds, 0.5, malfunction_rng="reference")
    got = eval_run(EmulEngine, rm, q, seeds, 0.5, malfunction_rng="reference")
    assert_same_episodes(got, want, name)
    assert (want[1]["num_malfunctions"] > 0).any()


def _learner(name, n_envs=4, **kw):
    rm = rail_map(name)
    env = EmulSwitchEnv(api.RailEnv(rm.fixture), max_steps=100_000, n_envs=n_envs, q_cap=1 << 16, **kw)
    m = api.DistrQLearning(env, **HP, default_q=0.5, seed=SEED0)
    m.learn(2, None, 0)
    return env, m


@pytest.mark.parametrize("malfunction_rng", ["philox", "reference"])
def test_emul_evaluate_equals_load_and_test_and_leaves_the_learner_alone(malfunction_rng):
    env, m = _learner("slips24_t6", malfunction_rng=malfunction_rng)
    q = m.q_table
    state = env.engine.buf["state"].clone()
    q_copy = {k: list(v) for k, v in q.items()}
    cum, arr, delays, malf, at_dest = m.evaluate()
    assert np.array_equal(env.engine.buf["state"], state), "evaluate() wrote to the learner's engine"
    assert m.q_table == q_copy
    # the reference's eval.py: load() the saved table into a learner of as many environments, then test()
    with tempfile.TemporaryDirectory() as tmp:
        m.save(os.path.join(tmp, "q.pkl"))
        env2 = EmulSwitchEnv(api.RailEnv(env.rail_map.fixture), max_steps=100_000, n_envs=4, q_cap=1 << 16, malfunction_rng=malfunction_rng)
        m2 = api.DistrQLearning(env2, **HP, default_q=0.5, seed=SEED0)
        m2.load(os.path.join(tmp, "q.pkl"))
    wc, wa, wd = m2.test(None, save_outputs=False, _batched=True)
    _, log, _ = env2.engine.episode_log()
    assert np.array_equal(cum, wc) and np.array_equal(arr, wa) and np.array_equal(delays, wd)
    assert np.array_equal(malf, log["num_malfunctions"][:, 0])
    T = env.rail_map.trains.T
    assert at_dest == [backend.train_set(r["arrived_mask"], r["arrived_mask_hi"], T) for r in log[:, 0]]
    assert [len(a) for a in at_dest] == list(arr)
    # more runs than the learner has environments, explicit seeds, the batched file
    with tempfile.TemporaryDirectory() as tmp:
        r = m.evaluate(n_runs=9, out_dir=tmp)
        z = np.load(os.path.join(tmp, "eval_batched.npz"))
        assert np.array_equal(z["cum_reward"], r[0]) and np.array_equal(z["seeds"], np.arange(9) + SEED0)
    assert np.array_equal(r[0][:4], cum)
    r2 = m.evaluate(seeds=[SEED0 + 2, SEED0])
    assert list(r2[0]) == [cum[2], cum[0]]


def test_vectorised_dict_conversion_equals_obs_to_key():
    for name in ("slips24_t6", "t100"):
        rm = rail_map(name)
        q = table(name, "init", 0.0)
        a_max = int(max(rm.tab.sw_A))
        keys, vals = rm.q_arrays(q, a_max)
        assert list(keys) == [rm.obs_to_key(o) for o in q]
        for (o, row), v in zip(q.items(), vals):
            assert list(v[:len(row)]) == row and not v[len(row):].any()
    with pytest.raises(ValueError, match="not one of this map's states"):
        rail_map("slips24_t6").q_arrays({(0, 0, 1, 1, 0, 0, 0, 0, 0, -1): [0.0, 0.0]}, 3)


def test_eval_context_layout_and_sizes():
    lib = backend.load_library(build_emul())
    rm = rail_map("c4_rail100_t50")
    cfg = backend.Config(n_envs=8192, q_cap=262144, pend_cap=8, max_steps=100000, ep_cap=1)
    private, ev = backend.Sizes(), backend.Sizes()
    assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(private)) == 0
    cfg.q_cap, cfg.eval_q = 131072, 1
    assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(ev)) == 0
    assert private.eval_q_bytes == 0 and ev.eval_q_bytes == 131072 * ev.q_stride * 8
    assert private.env_stride - ev.env_stride >= 262144 * private.q_stride * 8 - 128   # no Q region
    assert ev.env_stride % 128 == 0 and ev.env_stride < private.env_stride // 100 and ev.state_bytes == 8192 * ev.env_stride
    cfg.eval_q = 2
    assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(ev)) == -1
    assert b"eval_q must be 0 or 1" in lib.sfl_last_error()


def test_abi_version_and_appended_offsets():
    assert backend.load_library(build_emul()).sfl_abi_version() == backend.ABI_VERSION == 10
    fields = [("sfl_config", "malf_rng"), ("sfl_config", "eval_q"), ("sfl_sizes", "rng_offset"), ("sfl_sizes", "eval_q_bytes"),
              ("sfl_buffers", "shared_c"), ("sfl_buffers", "eval_q")]
    prog = "#include <stdio.h>\n#include <stddef.h>\n#include \"switchfl_b200.h\"\nint main(void) {\n" + "".join(
        f'  printf("%zu\\n", offsetof({s}, {f}));\n' for s, f in fields) + \
        '  printf("%zu %zu %zu\\n", sizeof(sfl_config), sizeof(sfl_sizes), sizeof(sfl_buffers));\n  return 0;\n}\n'
    with tempfile.TemporaryDirectory() as tmp:
        open(os.path.join(tmp, "o.c"), "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(tmp, "o"), os.path.join(tmp, "o.c")])
        got = [int(x) for x in subprocess.check_output([os.path.join(tmp, "o")]).split()]
    cls = {"sfl_config": backend.Config, "sfl_sizes": backend.Sizes, "sfl_buffers": backend.Buffers}
    want = [getattr(cls[s], f).offset for s, f in fields]
    assert got[:len(fields)] == want
    # every earlier field keeps its offset: the new ones are the last of their structs
    assert want == [48, 52, 128, 136, 104, 112]
    assert got[len(fields):] == [C.sizeof(backend.Config), C.sizeof(backend.Sizes), C.sizeof(backend.Buffers)] == [56, 144, 120]


def test_loud_refusals():
    rm = rail_map("slips24_t6")
    with pytest.raises(RuntimeError, match="no shared-table mode"):
        EmulEngine(rm, n_envs=2, q_cap=1024, eval_q=True, shared_q=True)
    with pytest.raises(RuntimeError, match="greedy rollouts only"):
        EmulEngine(rm, n_envs=2, q_cap=1024, eval_q=True, rng="reference")
    with pytest.raises(RuntimeError, match="no instrumented kernel"):
        EmulEngine(rm, n_envs=2, q_cap=1024, eval_q=True, phase_clock=True)
    q = table("slips24_t6", "init", 0.0)
    assert len(q) > 512
    eng = EmulEngine(rm, n_envs=2, q_cap=512, eval_q=True, act_cap=4, ev_cap=4, dec_cap=0)
    eng.set_hparams(**HP, episodes=1)
    eng.reset()
    eng.set_eval_table({k: q[k] for k in list(q)[:511]})
    for mode in (backend.MODE_LEARN, backend.MODE_REPLAY, backend.MODE_STEP):
        with pytest.raises(RuntimeError, match="SFL_MODE_GREEDY only"):
            eng.run(mode, 8)
    with pytest.raises(RuntimeError, match="per-environment tables"):
        eng.reapply_q_init()
    with pytest.raises(RuntimeError, match="per-environment tables"):
        eng.import_q(0, q)
    with pytest.raises(RuntimeError, match="per-environment tables"):
        eng.q_rows(0)
    with pytest.raises(RuntimeError, match="error -3: the evaluation table needs q_cap above its row count"):
        eng.set_eval_table(q)
    keys, vals = rm.q_arrays({k: q[k] for k in list(q)[:512]}, eng.sizes.a_max)
    keys[511] = keys[0]                                  # n_rows counts rows, repeated keys or not
    u32, f64 = C.POINTER(C.c_uint32), C.POINTER(C.c_double)
    assert eng.lib.sfl_set_eval_table(eng.ctx, keys.ctypes.data_as(u32), vals.ctypes.data_as(f64), 512, None) == -3
    eng.run(backend.MODE_GREEDY, 8)
    eng.close()
    traced = EmulEngine(rm, n_envs=2, q_cap=1024, eval_q=True, dec_cap=16, tick_cap=16)
    traced.set_hparams(**HP, episodes=1)
    traced.reset()
    traced.set_eval_table(q)
    with pytest.raises(RuntimeError, match="no traced or instrumented kernel"):
        traced.run(backend.MODE_GREEDY, 8)
    traced.close()
    private = EmulEngine(rm, n_envs=2, q_cap=1024)
    with pytest.raises(RuntimeError, match=r"Engine\(eval_q=True\)"):
        private.set_eval_table(q)
    lib = private.lib
    with pytest.raises(RuntimeError, match="not created as an evaluation context"):
        private._ck(lib.sfl_set_eval_table(private.ctx, None, None, 0, None))
    private.close()
    lib = backend.load_library(build_emul())
    cfg = backend.Config(n_envs=2, q_cap=1024, pend_cap=8, max_steps=100, ep_cap=1, eval_q=1)
    ctx = C.c_void_p()
    assert lib.sfl_create(C.byref(rm.desc), C.byref(cfg), 0, C.byref(ctx)) == 0
    sz = backend.Sizes()
    lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(sz))
    import torch
    bufs = {k: torch.zeros(max(int(n), 16), dtype=torch.uint8) for k, n in (("state", sz.state_bytes), ("hparams", sz.hparams_bytes),
                                                                          ("counters", sz.counters_bytes))}
    b = backend.Buffers(**{k: v.data_ptr() for k, v in bufs.items()})
    assert lib.sfl_bind(ctx, C.byref(b)) == -1 and b"needs the eval_q buffer" in lib.sfl_last_error()
    lib.sfl_destroy(ctx)


def test_cli_launch_eval_matches_the_per_environment_path():
    """The grid tree of the launcher test: launch_eval's eval_i/ arrays equal load() + test() on as many environments."""
    env_section = {"width": 18, "height": 18, "max_num_cities": 5, "max_rails_between_cities": 1, "max_rail_pairs_in_city": 1,
                   "number_of_agents": 2, "malfunction_rate": 0.05, "min_duration": 2, "max_duration": 5}
    with tempfile.TemporaryDirectory() as tmp:
        dirs = cli.launch_grid({"epsilon": [0.5, 0.1], "epsilon_decay_rate": [0.9997], "lr": [0.1], "lr_decay_rate": [1.0]},
                               random_seeds=[64], out_dir=tmp, env_section=env_section, num_episodes=3, checkpoint_freq=10 ** 9,
                               exploit_freq=None, env_cls=EmulSwitchEnv)
        res = cli.launch_eval(dirs, env_cls=EmulSwitchEnv)
        for d in dirs:
            # what launch_eval computed before evaluation contexts existed: ten private tables, one test()
            import configparser
            config = configparser.ConfigParser()
            config.read(os.path.join(d, "config.ini"))
            envs, mdl, seed = config["ENV"], config["MODEL"], int(config["MISC"]["random_seed"])
            mf = api.ParamMalfunctionGen(api.MalfunctionParameters(float(envs["malfunction_rate"]), int(envs["min_duration"]),
                                                                   int(envs["max_duration"])))
            env = EmulSwitchEnv(api.RailEnv(cli.fixture_from_env_section(dict(envs), seed), malfunction_generator=mf),
                                max_steps=100_000, n_envs=10)
            m = api.DistrQLearning(env, gamma=float(mdl["gamma"]), epsilon=float(mdl["epsilon"]),
                                   epsilon_decay_rate=float(mdl["epsilon_decay_rate"]), lr=float(mdl["lr"]),
                                   lr_decay_rate=float(mdl["lr_decay_rate"]), default_q=float(mdl["default_q"]), seed=seed)
            m.load(os.path.join(d, "distr_q_model.pkl"))
            cum, arrived, delays = m.test(out_dir=None, plot=False, save_outputs=False, _batched=True)
            assert np.array_equal(res[d], np.stack([cum, arrived]))
            for i in range(10):
                assert np.array_equal(np.load(os.path.join(d, f"eval_{i}", "cum_reward.npz"))["x"], cum[i])
                assert np.array_equal(np.load(os.path.join(d, f"eval_{i}", "delays.npz"))["x"], np.array(list(delays[i])))
            assert not os.path.exists(os.path.join(d, f"eval_10")) and not os.path.exists(os.path.join(d, "eval_batched.npz"))
            env.engine.close()
        many = cli.launch_eval(dirs[:1], env_cls=EmulSwitchEnv, num_evals=64)[dirs[0]]
        z = np.load(os.path.join(dirs[0], "eval_batched.npz"))
        assert many.shape == (2, 64) and z["cum_reward"].shape == (64,) and z["delays"].shape == (64, 2)
        assert np.array_equal(z["cum_reward"], many[0]) and np.array_equal(z["arrived_trains"], many[1])
        assert np.array_equal(z["seeds"], np.arange(64) + 64) and np.array_equal(many[:, :10], res[dirs[0]])
        assert not os.path.exists(os.path.join(dirs[0], "eval_10"))


def test_cli_flag_num_evals(monkeypatch):
    seen = {}
    monkeypatch.setattr(cli, "launch_eval", lambda dirs, **kw: seen.update(dirs=dirs, **kw))
    cli.main(["--eval", "a", "b", "--num-evals", "64"])
    assert seen["dirs"] == ["a", "b"] and seen["num_evals"] == 64
    with pytest.raises(SystemExit):
        cli.main([])                                     # learning still needs -c


# ---------------------------------------------------------------------------------------------- GPU
ONE_WORD_LANES = (1, 2, 4, 8, 16, 32)
GPU_CASES = ([(name, lanes) for name in ("c1_synth18", "slips24_t6", "c3_rail80_s64", "c4_rail100_t50")
              for lanes in ONE_WORD_LANES] +
             [("t100", lanes) for lanes in (8, 16, 32)])
# bench_eval.py's batches: (map, environments)
BENCH_BATCHES = (("c4", 8192), ("c4", 32768), ("t100", 3552), ("t100", 8192), ("t100", 32768))


def _parity_variants(cls=backend.Engine):
    out = set()
    for name, lanes in GPU_CASES:
        eng = cls(rail_map(name), n_envs=6, q_cap=1 << 17, ep_cap=1, eval_q=True, lanes=lanes, bind=False)
        out.add(eng.kernel_variant(backend.MODE_GREEDY))
        eng.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,lanes", GPU_CASES)
def test_cuda_eval_kernel_equals_private_tables(name, lanes):
    rm = rail_map(name)
    q = table(name, "holes", 0.5)
    seeds = np.arange(6) + SEED0
    want = private_run(EmulEngine, rm, q, seeds, 0.5)
    got = eval_run(backend.Engine, rm, q, seeds, 0.5, lanes=lanes)
    assert "EVQ=1" in got[3] and f"G={lanes}," in got[3]
    assert_same_episodes(got, want, (name, lanes))
    if lanes == 8:
        got = eval_run(backend.Engine, rm, q, seeds, 0.5, lanes=lanes, malfunction_rng="reference")
        assert_same_episodes(got, private_run(EmulEngine, rm, q, seeds, 0.5, malfunction_rng="reference"), (name, "reference"))


def test_gpu_cases_cover_every_lane_width_and_staging_plan():
    """Which k_eval instantiations the GPU cases below run (the launch plan is host code: the host build names them too):
    every lane width, the tail staged and in HBM, one pass and chunked, and the three NW = 2 kernels."""
    v = _parity_variants(EmulEngine)
    for G in ONE_WORD_LANES:
        assert any(x.startswith(f"k_eval<G={G},") and ",NW=2" not in x for x in v), G
    for th, one in (("TH=0", "ONE=0"), ("TH=0", "ONE=1"), ("TH=1", "ONE=1")):
        assert any(th in x and one in x for x in v), (th, one)
    assert sorted(x.split(",")[0] for x in v if ",NW=2" in x) == ["k_eval<G=16", "k_eval<G=32", "k_eval<G=8"]
    assert all(x.endswith("EVQ=1>") for x in v)


@pytest.mark.gpu
def test_cuda_bench_eval_variants_are_parity_tested():
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import bench_eval
    tested = _parity_variants()
    for name, n in BENCH_BATCHES:
        rm = bench_eval.rail_map(name)
        eng = backend.Engine(rm, n_envs=n, q_cap=1 << 17, ep_cap=1, eval_q=True, bind=False)
        variant = eng.kernel_variant(backend.MODE_GREEDY)
        eng.close()
        assert variant in tested, (name, n, variant, sorted(tested))
    assert {(name, n) for name, n in BENCH_BATCHES} == {(m, n) for m, ns in bench_eval.BATCHES.items() for n in ns}


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", [("c4_rail100_t50", 8192), ("t100", 3552)])
def test_cuda_eval_kernel_at_the_bench_batch(name, n):
    """The bench batch on the device against the host build on a subset of its environments (results depend on the seed only)."""
    rm = rail_map(name)
    q = table(name, "init", 0.5)
    seeds = np.arange(n) + SEED0
    got = eval_run(backend.Engine, rm, q, seeds, 0.5)
    pick = np.arange(0, n, n // 12)
    want = private_run(EmulEngine, rm, q, seeds[pick], 0.5)
    assert_same_episodes((got[0][pick], got[1][pick], got[2][pick]), want, (name, n))
    assert (got[1]["arrived"] > 0).all()
