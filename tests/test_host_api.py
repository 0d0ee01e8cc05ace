"""CPU: the host layer -- C-ABI surface, struct layouts, the drop-in classes' outputs, multi-process sharding (gloo).

No compute call is made on the product library here (there is no GPU); the drop-in classes are exercised on the
test-only host build of the device sources (tests/emul)."""
import ctypes as C
import os
import pickle
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import __graft_entry__ as entry
from switchfl_b200 import api, backend, mapgen, sharding
from tests._util import load_golden
from tests.emulated import EmulEngine, EmulSwitchEnv, build_emul

ROOT = entry.ROOT
HEADER = os.path.join(ROOT, "include", "switchfl_b200.h")


@pytest.fixture(scope="module")
def product_lib():
    entry.build()                       # nvcc cross-compiles without a GPU; on the GPU box the prebuilt .so is current
    return C.CDLL(entry.LIB)


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sfl_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(product_lib):
    names = declared_functions()
    assert {"sfl_create", "sfl_run", "sfl_reset", "sfl_bind", "sfl_export_q", "sfl_import_q", "sfl_query_sizes"} <= set(names)
    for n in names:
        assert hasattr(product_lib, n), f"{n} declared in include/switchfl_b200.h but not exported"
    assert product_lib.sfl_abi_version() == backend.ABI_VERSION


def test_struct_layouts_match_the_header():
    """ctypes / numpy mirrors in backend.py against sizeof() as the C compiler sees the header."""
    prog = r'''
#include <stdio.h>
#include "switchfl_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(sfl_map_desc), sizeof(sfl_config), sizeof(sfl_hparams), sizeof(sfl_sizes),
         sizeof(sfl_buffers), sizeof(sfl_env_counters), sizeof(sfl_dec_rec), sizeof(sfl_tick_rec), sizeof(sfl_ep_rec), sizeof(sfl_step_rec));
  return 0;
}'''
    with tempfile.TemporaryDirectory() as tmp:
        open(os.path.join(tmp, "s.c"), "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(tmp, "s"), os.path.join(tmp, "s.c")])
        got = [int(x) for x in subprocess.check_output([os.path.join(tmp, "s")]).split()]
    want = [C.sizeof(backend.MapDesc), C.sizeof(backend.Config), backend.HPARAMS_DT.itemsize, C.sizeof(backend.Sizes),
            C.sizeof(backend.Buffers), backend.COUNTERS_DT.itemsize, backend.DEC_DT.itemsize, backend.TICK_DT.itemsize,
            backend.EP_DT.itemsize, backend.STEP_DT.itemsize]
    assert got == want


def test_query_sizes_and_loud_failure_without_gpu(product_lib):
    import torch
    fx, _ = load_golden("c1_synth18")
    rm = backend.RailMap(fx)
    lib = backend.load_library()
    cfg = backend.Config(n_envs=4096, q_cap=1024, pend_cap=8, max_steps=100000, dec_cap=0, tick_cap=0, ep_cap=4, act_cap=0, ev_cap=0, trace_sem=0)
    sz = backend.Sizes()
    assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(sz)) == 0
    assert sz.env_stride % 128 == 0 and sz.state_bytes == 4096 * sz.env_stride
    assert sz.a_max == int(max(rm.tab.sw_A)) and sz.q_stride == sz.a_max + 1
    assert sz.env_stride >= 1024 * sz.q_stride * 8
    cfg.q_cap = 1000                                             # not a power of two
    assert lib.sfl_query_sizes(C.byref(rm.desc), C.byref(cfg), C.byref(sz)) == -1
    assert b"power of two" in lib.sfl_last_error()
    if not torch.cuda.is_available():
        cfg.q_cap = 1024
        ctx = C.c_void_p()
        assert lib.sfl_create(C.byref(rm.desc), C.byref(cfg), 0, C.byref(ctx)) == -2      # SFL_E_CUDA: no CPU path
        assert b"no CPU path" in lib.sfl_last_error()
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            backend.Engine(rm, n_envs=4)


def test_product_package_never_touches_the_oracle():
    pkg = os.path.join(ROOT, "network-distributed-q-learning_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "libsfl_emul" not in src, f


def test_key_obs_roundtrip_and_naming():
    fx, g = load_golden("slips24_t6")
    rm = backend.RailMap(fx)
    for obs in g["dec_obs"][:200]:
        o = tuple(int(x) for x in obs if x != -9)
        assert rm.key_to_obs(rm.obs_to_key(o)) == o
    # utils/naming.py:27-60 docstring examples: (4, 3) <-> 'switch_4-3'
    assert all(re.fullmatch(r"switch_\d+-\d+", n) for n in rm.tab.switch_names())
    assert rm.tab.switch_names() == sorted(rm.tab.switch_names(), key=lambda n: tuple(int(x) for x in n[7:].split("-")))


def test_drop_in_learn_outputs_have_the_reference_layout():
    """main.py:51-66 against the drop-in classes (host build of the kernels): files, names, pkl dict layout."""
    emul = build_emul()
    fx, _ = load_golden("c1_synth18")
    rail_env = api.RailEnv(fx, malfunction_generator=api.ParamMalfunctionGen(api.MalfunctionParameters(0.01, 5, 15)))
    env = EmulSwitchEnv(rail_env, render_mode=None, max_steps=100_000, n_envs=3, q_cap=1024, ep_cap=4)
    assert env.possible_agents == env.rail_map.tab.switch_names()
    model = api.DistrQLearning(env=env, gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0, seed=450565)
    with tempfile.TemporaryDirectory() as out:
        model.learn(num_episodes=6, out_dir=out, checkpoint_freq=3, exploit_freq=2)
        model.save(os.path.join(out, "distr_q_model.pkl"))
        for name in ("cum_reward", "arrived_trains", "delays", "num_malfunctions", "trains_at_dest", "cum_reward_exploit", "arrived_trains_exploit",
                     "cum_reward_checkpoint_3", "arrived_trains_checkpoint_3", "delays_checkpoint_3", "trains_at_dest_checkpoint_3",
                     "num_malfunctions_checkpoint_3"):
            with np.load(os.path.join(out, name + ".npz")) as z:
                assert z.files == ["x"], name                                  # distr_q.py:290-294, 368-375: key is always "x"
        assert np.load(os.path.join(out, "cum_reward.npz"))["x"].shape == (6,)
        assert np.load(os.path.join(out, "delays.npz"))["x"].shape == (6, 2)
        assert len(np.load(os.path.join(out, "cum_reward_exploit.npz"))["x"]) == 3     # before episodes t = 1, 3, 5 ((t+1) % 2 == 0), :277-280
        assert os.path.exists(os.path.join(out, "checkpoint_3.pkl"))
        q = pickle.load(open(os.path.join(out, "distr_q_model.pkl"), "rb"))
        assert isinstance(q, dict) and len(q) > 0
        tab = env.rail_map.tab
        for k, v in q.items():
            s = tab.switch_cells.index((int(k[0]), int(k[1])))
            P, A = int(tab.sw_P[s]), int(tab.sw_A[s])
            assert isinstance(k, tuple) and len(k) == 2 + 4 * P and all(isinstance(x, np.int64) for x in k)   # observer.py:303-306
            assert isinstance(v, list) and len(v) == A and all(isinstance(x, float) for x in v)                # distr_q.py:57
        # load() -> the same table comes back out of the engine
        model2 = api.DistrQLearning(env=env, gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)
        model2.load(os.path.join(out, "distr_q_model.pkl"))
        assert env.engine.export_q(1) == {tuple(int(x) for x in k): v for k, v in q.items()}
        r, arrived, delays = model2.test(out_dir=None, save_outputs=False)
        assert isinstance(r, float) and 0 <= arrived <= 2 and len(delays) == 2
    with pytest.raises(AttributeError):
        model.save("x.csv", mode="csv")                                        # distr_q.py:505-508


# ---------------------------------------------------------------------------------------------- sharding (gloo, world size 2)
def test_shard_range_partitions():
    for n in (1, 7, 4096, 65536):
        for ws in (1, 2, 3, 8):
            r = [sharding.shard_range(n, k, ws) for k in range(ws)]
            assert r[0][0] == 0 and r[-1][1] == n and all(r[i][1] == r[i + 1][0] for i in range(ws - 1))
            assert max(b - a for a, b in r) - min(b - a for a, b in r) <= 1


def test_grid_points_follow_hyperparam_tuning_order():
    g = sharding.grid_points({"epsilon": [0.5, 0.3], "lr": [0.1]}, seeds=[64, 65, 66])        # hyperparam_tuning.py:10-48
    assert list(g["epsilon"]) == [0.5, 0.5, 0.5, 0.3, 0.3, 0.3] and list(g["seeds"]) == [64, 65, 66, 64, 65, 66]


_WORKER = r'''
import os, sys, json
import numpy as np
sys.path.insert(0, sys.argv[1])
from __graft_entry__ import load_package
load_package()
import torch.distributed as dist
from switchfl_b200 import backend, mapgen, sharding
from tests.emulated import EmulEngine
rank, ws, _ = sharding.world()
dist.init_process_group("gloo", rank=rank, world_size=ws)
fx = mapgen.load_fixture(os.path.join(sys.argv[1], "tests", "golden", "c1_synth18.fixture.npz"))
rm = backend.RailMap(fx)
grid = sharding.grid_points({"epsilon": [0.5, 0.2], "lr": [0.1]}, seeds=[64, 65, 66])
mine = sharding.shard_grid(grid, rank, ws)
n = len(mine["seeds"])
eng = EmulEngine(rm, n_envs=n, q_cap=1024, ep_cap=4)
eng.set_hparams(gamma=1.0, epsilon=mine["epsilon"], epsilon_decay_rate=0.9997, lr=mine["lr"], lr_decay_rate=1.0, default_q=0.0,
                seeds=mine["seeds"], episodes=3)
eng.reset(); eng.enable_q_init(True)
eng.run(backend.MODE_LEARN, 100000)
eng.check_errors()
c = eng.counters()
times, counts = sharding.reduce_run(dist, [10.0 + rank], [int(c["decisions"].sum()), int(c["ticks"].sum()), n])
_, log, _ = eng.episode_log()
allm = sharding.gather_metrics(dist, np.ascontiguousarray(log["cum_reward"][:, :3]))
if rank == 0:
    print("RESULT " + json.dumps({"times": times, "counts": counts, "cum": allm.tolist()}))
dist.destroy_process_group()
'''


def test_two_ranks_shard_the_grid_and_reduce_like_one_process():
    import json
    emul = build_emul()
    fx, _ = load_golden("c1_synth18")
    rm = backend.RailMap(fx)
    grid = sharding.grid_points({"epsilon": [0.5, 0.2], "lr": [0.1]}, seeds=[64, 65, 66])
    eng = EmulEngine(rm, n_envs=6, q_cap=1024, ep_cap=4)
    eng.set_hparams(gamma=1.0, epsilon=grid["epsilon"], epsilon_decay_rate=0.9997, lr=grid["lr"], lr_decay_rate=1.0, default_q=0.0,
                    seeds=grid["seeds"], episodes=3)
    eng.reset(); eng.enable_q_init(True)
    eng.run(backend.MODE_LEARN, 100000)
    c = eng.counters()
    _, log, _ = eng.episode_log()
    with tempfile.TemporaryDirectory() as tmp:
        w = os.path.join(tmp, "w.py")
        open(w, "w").write(_WORKER)
        out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                              "--master-port", "29541", w, ROOT, emul], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    res = json.loads([l for l in out.stdout.splitlines() if l.startswith("RESULT ")][0][7:])
    assert res["times"] == [11.0]                                                        # MAX over ranks
    assert res["counts"] == [int(c["decisions"].sum()), int(c["ticks"].sum()), 6]        # SUM over ranks == single process
    assert np.array_equal(np.array(res["cum"]), log["cum_reward"][:, :3])                # env i gives the same curve on any rank


# ---------------------------------------------------------------------------------------------- driver scripts (main.py / hyperparam_tuning.py)
def _write_ini(path, out_dir, fixture=None, **model):
    import configparser
    c = configparser.ConfigParser()
    c["MISC"] = {"random_seed": 450565, "out_dir": out_dir, "checkpoint_freq": 2, "exploit_freq": 2, "n_envs": 2}
    c["ENV"] = {"width": 18, "height": 18, "max_num_cities": 5, "max_rails_between_cities": 1, "max_rail_pairs_in_city": 1,
                "number_of_agents": 2, "malfunction_rate": 0.01, "min_duration": 5, "max_duration": 15}
    if fixture:
        c["ENV"]["fixture"] = fixture
    c["MODEL"] = {"gamma": 1.0, "epsilon": 0.5, "epsilon_decay_rate": 0.9997, "lr": 0.1, "lr_decay_rate": 1.0, "default_q": 0.0,
                  "num_episodes": 4, **model}
    with open(path, "w") as f:
        c.write(f)


def test_cli_runs_the_reference_ini(capsys):
    """main.py:13-78 with the reference's config.ini schema (hyperparam_tuning.py:51-78)."""
    from switchfl_b200 import cli
    emul = build_emul()
    with tempfile.TemporaryDirectory() as tmp:
        ini = os.path.join(tmp, "config.ini")
        _write_ini(ini, os.path.join(tmp, "out"), fixture=os.path.join(ROOT, "tests", "golden", "c1_synth18.fixture.npz"))
        model = cli.launch_experiment(ini, env_cls=EmulSwitchEnv)
        out = capsys.readouterr().out
        for line in ("DONE!", "TOTAL TIME:", "Seconds per episode:", "Flatland step time:", "Total step time:", "Total last time:",
                     "Action selection time:", "Update time:", "Flatland reset time:", "Total reset time:"):          # main.py:68-78
            assert line in out
        assert os.path.exists(os.path.join(tmp, "out", "distr_q_model.pkl")) and os.path.exists(os.path.join(tmp, "out", "checkpoint_2.pkl"))
        assert model.metrics["cum_reward"].shape == (2, 4)
        # without ENV.fixture the synthetic generator builds a map of the requested size / train count
        _write_ini(ini, os.path.join(tmp, "out2"))
        m2 = cli.launch_experiment(ini, env_cls=EmulSwitchEnv)
        assert m2.env.rail_env.width == 18 and m2.env.rail_env.get_num_agents() == 2


def test_grid_launcher_writes_the_reference_tree():
    """hyperparam_tuning.py:42-91: exp_i/seed_j/config.ini + outputs; grid points are the env axis of one engine."""
    import configparser
    from switchfl_b200 import cli
    emul = build_emul()
    env_section = {"width": 18, "height": 18, "max_num_cities": 5, "max_rails_between_cities": 1, "max_rail_pairs_in_city": 1,
                   "number_of_agents": 2, "malfunction_rate": 0.0, "min_duration": 0, "max_duration": 0}
    with tempfile.TemporaryDirectory() as tmp:
        dirs = cli.launch_grid({"epsilon": [0.5, 0.1], "epsilon_decay_rate": [0.9997], "lr": [0.1], "lr_decay_rate": [1.0]},
                               random_seeds=[64, 65], out_dir=tmp, env_section=env_section, num_episodes=3, checkpoint_freq=10 ** 9,
                               exploit_freq=None, env_cls=EmulSwitchEnv)
        assert sorted(os.path.relpath(d, tmp) for d in dirs) == ["exp_0/seed_0", "exp_0/seed_1", "exp_1/seed_0", "exp_1/seed_1"]
        res = cli.launch_eval(dirs[:2], env_cls=EmulSwitchEnv)                       # eval.py:31-97
        for d in dirs[:2]:
            assert res[d].shape == (2, 1) and np.load(os.path.join(d, "eval_0", "cum_reward.npz"))["x"].shape == ()
            assert len(np.load(os.path.join(d, "eval_0", "delays.npz"))["x"]) == 2
        for d in dirs:
            c = configparser.ConfigParser()
            c.read(os.path.join(d, "config.ini"))
            assert set(c["MODEL"]) == {"gamma", "epsilon", "epsilon_decay_rate", "lr", "lr_decay_rate", "default_q", "num_episodes"}
            assert np.load(os.path.join(d, "cum_reward.npz"))["x"].shape == (3,)
            assert isinstance(pickle.load(open(os.path.join(d, "distr_q_model.pkl"), "rb")), dict)


# ---------------------------------------------------------------------------------------------- shared-table mode (extension)
HP_SHARED = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0, default_q=0.0)


def _shared_run(rm, emul, seeds, launches=5, ticks=64, dist=None, overlapped=False, cls=None):
    eng = (cls or EmulEngine)(rm, n_envs=len(seeds), q_cap=2, ep_cap=4, shared_q=True)
    eng.set_hparams(**HP_SHARED, seeds=seeds, episodes=-1)
    eng.reset()
    eng.init_shared_q(0.0)
    for _ in range(launches):
        if overlapped:                                   # two tables / accumulator pairs, TD steps folded in one step late
            eng.run_shared(ticks, dist)
        else:
            eng.run(backend.MODE_LEARN, ticks)
            eng.shared_q_sync(dist)
        eng.check_errors()
    if overlapped:
        eng.shared_q_flush()
    return eng


def test_shared_table_mode_is_deterministic_and_averages():
    """No reference counterpart (BASELINE config 5): properties of the policy stated in DESIGN.md.  Integer
    accumulation makes the result independent of the order in which environments arrive; N identical environments
    propose N identical steps whose mean is the step, so they leave the table a single environment leaves."""
    emul = build_emul()
    fx, _ = load_golden("slips24_t6")
    rm = backend.RailMap(fx)
    one = _shared_run(rm, emul, [7])
    q1 = one.shared_q_table()
    assert np.array_equal(q1, _shared_run(rm, emul, [7]).shared_q_table())
    assert np.array_equal(q1, _shared_run(rm, emul, [7, 7, 7, 7]).shared_q_table())
    mixed = _shared_run(rm, emul, [1, 2, 3, 4, 5, 6])
    qm = mixed.shared_q_table()
    assert np.isfinite(qm).all() and not np.array_equal(qm, q1)
    init = EmulEngine(rm, n_envs=1, q_cap=2, shared_q=True)
    init.init_shared_q(0.0)
    q0 = init.shared_q_table()
    assert set(np.unique(q0)) <= {0.0, 500.0, 1000.0} and (q0 == 500.0).any()             # distr_q.py:44-45, 156-181
    learned = mixed.export_q(0)
    assert learned and all(len(k) in (14, 18) for k in learned)
    # the environments keep no private rows in this mode
    assert (mixed.counters()["q_rows"] == 0).all()


def test_shared_table_overlapped_schedule_properties():
    """run_shared (double-buffered tables, synchronisation one step late): deterministic, N identical environments leave
    the table one leaves, and the delay really changes the trajectory (it is not the synchronous schedule in disguise)."""
    emul = build_emul()
    fx, _ = load_golden("slips24_t6")
    rm = backend.RailMap(fx)
    q1 = _shared_run(rm, emul, [7], overlapped=True).shared_q_table()
    assert np.array_equal(q1, _shared_run(rm, emul, [7], overlapped=True).shared_q_table())
    assert np.array_equal(q1, _shared_run(rm, emul, [7, 7, 7], overlapped=True).shared_q_table())
    mixed = _shared_run(rm, emul, [1, 2, 3, 4, 5, 6], overlapped=True)
    qm = mixed.shared_q_table()
    assert np.isfinite(qm).all() and not np.array_equal(qm, q1)
    assert not np.array_equal(qm, _shared_run(rm, emul, [1, 2, 3, 4, 5, 6]).shared_q_table())
    # a further run continues from the flushed table on both buffers
    mixed.run_shared(64)
    mixed.shared_q_flush()
    assert np.isfinite(mixed.shared_q_table()).all() and (mixed.buf["shared_c"].numpy() == 0).all()


_SHARED_WORKER = r'''
import os, sys, json
import numpy as np
sys.path.insert(0, sys.argv[1])
from __graft_entry__ import load_package
load_package()
import torch.distributed as dist
from switchfl_b200 import backend, mapgen, sharding
sys.path.insert(0, os.path.join(sys.argv[1]))
from tests.test_host_api import _shared_run
rank, ws, _ = sharding.world()
dist.init_process_group("gloo", rank=rank, world_size=ws)
fx = mapgen.load_fixture(os.path.join(sys.argv[1], "tests", "golden", "slips24_t6.fixture.npz"))
rm = backend.RailMap(fx)
lo, hi = sharding.shard_range(6, rank, ws)
eng = _shared_run(rm, sys.argv[2], list(range(1 + lo, 1 + hi)), dist=dist, overlapped=len(sys.argv) > 4)
np.save(os.path.join(sys.argv[3], f"q{rank}.npy"), eng.shared_q_table())
dist.destroy_process_group()
'''


@pytest.mark.parametrize("overlapped", [False, True])
def test_shared_table_two_ranks_allreduce_equals_one_process(overlapped):
    """Two ranks with three environments each, accumulators all-reduced (gloo) before every apply: both ranks end with
    the table one process with all six environments ends with, bit for bit -- on the synchronous and on the overlapped
    (one step late) schedule."""
    emul = build_emul()
    fx, _ = load_golden("slips24_t6")
    rm = backend.RailMap(fx)
    want = _shared_run(rm, emul, [1, 2, 3, 4, 5, 6], overlapped=overlapped).shared_q_table()
    with tempfile.TemporaryDirectory() as tmp:
        w = os.path.join(tmp, "w.py")
        open(w, "w").write(_SHARED_WORKER)
        out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                              "--master-port", "29543" if not overlapped else "29545", w, ROOT, emul, tmp] + (["overlapped"] if overlapped else []),
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        q0, q1 = np.load(os.path.join(tmp, "q0.npy")), np.load(os.path.join(tmp, "q1.npy"))
    assert np.array_equal(q0, q1) and np.array_equal(q0, want)


def test_learn_does_not_depend_on_the_episode_log_capacity():
    """learn() cuts a run into ep_cap-sized launches with an sfl_reset in between; RailNetwork.reset (rail_network.py:135-149)
    never clears _train_prev_port / _train_source_port, so neither does a reset that continues a run: one episode per launch
    gives exactly what one launch for all episodes gives (metrics, Q-table)."""
    fx, _ = load_golden("slips24_t6")
    out = []
    for cap in (1, 16):
        env = EmulSwitchEnv(api.RailEnv(fx), render_mode=None, max_steps=100_000, n_envs=3, q_cap=4096, ep_cap=cap)
        m = api.DistrQLearning(env=env, gamma=0.95, epsilon=0.5, epsilon_decay_rate=0.999, lr=0.2, lr_decay_rate=1.0, default_q=0.0, seed=5)
        m.learn(num_episodes=7, out_dir=None, checkpoint_freq=0)
        out.append(m)
    a, b = out
    for k in ("cum_reward", "arrived_trains", "delays", "num_malfunctions"):
        assert np.array_equal(a.metrics[k], b.metrics[k]), k
    assert a.q_table == b.q_table and len(a.q_table) > 0


def test_learn_concurrently_equals_learning_in_turn():
    """api.learn_concurrently (hyperparam_tuning.py's fan-out on streams / threads): same metrics and Q-tables as learn() per
    model in turn."""
    fxs = [load_golden(n)[0] for n in ("c1_synth18", "slips24_t6", "loop_chord_7x7")]

    def models():
        out = []
        for k, fx in enumerate(fxs):
            env = EmulSwitchEnv(api.RailEnv(fx), render_mode=None, max_steps=100_000, n_envs=3, q_cap=4096, ep_cap=8)
            out.append(api.DistrQLearning(env=env, gamma=0.95, epsilon=0.5, epsilon_decay_rate=0.999, lr=0.2, lr_decay_rate=1.0, default_q=0.0, seed=50 + k))
        return out
    a, b = models(), models()
    for m in a:
        m.learn(num_episodes=5, out_dir=None, checkpoint_freq=0)
    api.learn_concurrently(b, 5)
    for x, y in zip(a, b):
        assert np.array_equal(x.metrics["cum_reward"], y.metrics["cum_reward"]) and np.array_equal(x.metrics["delays"], y.metrics["delays"])
        assert x.q_table == y.q_table and len(x.q_table) > 0


def test_bench_dump_outputs_are_reproducible_float64_and_what_the_engine_holds():
    """bench.py --dump-outputs (host build of the kernels): two runs on the same inputs write the same float64 files, and they
    hold the engine's counters and Q tables."""
    import bench
    rm = backend.RailMap(load_golden("c1_synth18")[0])
    dumps = []
    for _ in range(2):
        eng = EmulEngine(rm, n_envs=8, q_cap=1024, ep_cap=4)
        eng.set_hparams(**bench.HP, seeds=np.arange(8) + bench.SEED, episodes=-1)
        eng.reset()
        eng.enable_q_init(True)
        for _ in range(2):
            eng.run(backend.MODE_LEARN, 512)
        with tempfile.TemporaryDirectory() as tmp:
            bench.dump_outputs(tmp, [eng])
            dumps.append({f[:-len(".npy")]: np.load(os.path.join(tmp, f)) for f in os.listdir(tmp)})
    a, b = dumps
    assert a.keys() == b.keys()
    for k, v in a.items():
        assert v.dtype == np.float64 and np.isfinite(v).all() and np.array_equal(v, b[k]), k
    assert np.array_equal(a["counters_decisions"], eng.counters()["decisions"]) and a["counters_decisions"].min() > 0
    for env in range(8):
        mine = a["q_env"] == env
        q = {rm.key_to_obs(int(k)): [float(x) for x in v[:int(n)]]
             for k, n, v in zip(a["q_key"][mine], a["q_actions"][mine], a["q_val"][mine])}
        assert q == eng.export_q(env) and len(q) > 0
