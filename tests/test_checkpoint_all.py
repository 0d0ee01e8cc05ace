"""Checkpoints of every learner of a batch: the device-side compaction of many Q tables (``sfl_export_q_batch``,
``Engine.export_q_batch``), ``learn(env_out_dirs=...)`` with its overlapped writer, and the grid launcher's checkpoints.

``-m "not gpu"`` runs the host build of the device sources (tests/emul); ``-m gpu`` the CUDA compaction kernel."""
import ctypes as C
import os
import pickle
import tempfile
import threading
import time

import numpy as np
import pytest

from switchfl_b200 import api, backend, cli
from tests._util import load_golden
from tests.emulated import EmulEngine, EmulSwitchEnv

HP = dict(gamma=1.0, epsilon=0.5, epsilon_decay_rate=0.9997, lr=0.1, lr_decay_rate=1.0)
CKPT_NPZ = ("cum_reward", "arrived_trains", "delays", "trains_at_dest", "num_malfunctions")


def pkl_bytes(q) -> bytes:
    with tempfile.TemporaryDirectory() as tmp:
        api._dump_q(q, os.path.join(tmp, "q.pkl"))
        return open(os.path.join(tmp, "q.pkl"), "rb").read()


def learned(engine_cls, rm, n, episodes, default_q, q_cap=1024, ticks=512):
    """An engine whose environments learned ``episodes[i]`` episodes each (0: an empty table)."""
    eng = engine_cls(rm, n_envs=n, q_cap=q_cap, ep_cap=4)
    eng.set_hparams(**HP, default_q=default_q, seeds=np.arange(n) + 450565, episodes=episodes)
    eng.reset()
    eng.enable_q_init(True)
    while True:
        eng.run(backend.MODE_LEARN, ticks)
        c = eng.counters()
        if (c["halted"] == 1).all():
            return eng


def assert_same_export(eng, envs, include_init, default_q):
    got = eng.export_q_batch(envs, include_init=include_init, default_q=default_q)
    assert len(got) == len(envs)
    for q, i, d in zip(got, envs, np.broadcast_to(np.asarray(default_q, np.float64), (len(envs),))):
        want = eng.export_q(i, include_init=include_init, default_q=float(d))
        assert q == want and list(q) == list(want), (i, include_init)
        assert pkl_bytes(q) == pkl_bytes(want), (i, include_init)


@pytest.mark.parametrize("include_init", [False, True])
def test_batched_export_equals_the_single_export(include_init):
    fx, _ = load_golden("c1_synth18")
    rm = backend.RailMap(fx)
    dq = np.array([0.0, 0.5, -1.0, 0.5, 0.25])
    eng = learned(EmulEngine, rm, 5, [3, 0, 3, 2, 1], dq)
    rows = eng.counters()["q_rows"]
    assert rows[1] == 0 and (rows[[0, 2, 3, 4]] > 0).all()
    for lo, hi in [(0, 5), (1, 3), (4, 5), (1, 2), (2, 2)]:
        assert_same_export(eng, list(range(lo, hi)), include_init, dq[lo:hi])
    assert_same_export(eng, [3], include_init, 0.75)                     # one value for every environment
    none = eng.export_q_batch(range(5), include_init=include_init)       # default_q from the hparams
    assert none == [eng.export_q(i, include_init=include_init) for i in range(5)]
    with pytest.raises(ValueError):
        eng.export_q_batch([0, 2])
    eng.close()


def test_batched_export_of_a_full_table():
    """A table filled to q_cap - 1 rows (the kernel stops inserting there and flags SFL_ERR_Q_FULL)."""
    fx, _ = load_golden("c3_synth80_s64")
    rm = backend.RailMap(fx)
    eng = learned(EmulEngine, rm, 2, [1, 1], 0.0, q_cap=256, ticks=4096)
    assert (eng.counters()["q_rows"] == 255).all()
    assert_same_export(eng, [0, 1], True, 0.0)
    assert_same_export(eng, [1], False, 0.0)
    eng.close()


def test_refusals_and_corrupted_tables():
    fx, _ = load_golden("c1_synth18")
    rm = backend.RailMap(fx)
    eng = learned(EmulEngine, rm, 3, [2, 2, 2], 0.0)
    lib, ctx = eng.lib, eng.ctx
    off = np.array([0, 4, 8, 12], np.uint64)
    keys, vals, found = np.zeros(16, np.uint32), np.zeros(16 * eng.sizes.a_max), np.zeros(3, np.int32)
    p = lambda a: C.c_void_p(a.ctypes.data)

    def call(lo, hi, o=off, cap=16):
        return lib.sfl_export_q_batch(ctx, lo, hi, p(o), p(keys), p(vals), C.c_uint64(cap), p(found), None)

    for lo, hi in [(-1, 2), (0, 4), (2, 1)]:
        assert call(lo, hi) == -1 and b"bad environment range" in lib.sfl_last_error(), (lo, hi)
    assert call(0, 3, cap=11) == -3 and b"smaller than the last row offset" in lib.sfl_last_error()
    assert call(1, 2, o=off[2:], cap=11) == -3                          # the last offset of the range is what counts
    assert call(3, 3, o=off[3:], cap=12) == 0
    assert lib.sfl_export_q_batch(ctx, 0, 3, p(off), None, p(vals), C.c_uint64(16), p(found), None) == -1
    ev = EmulEngine(rm, n_envs=2, q_cap=1024, eval_q=True)
    assert ev.lib.sfl_export_q_batch(ev.ctx, 0, 2, p(off), p(keys), p(vals), C.c_uint64(16), p(found), None) == -4
    assert b"evaluation context" in ev.lib.sfl_last_error()
    with pytest.raises(RuntimeError, match="evaluation context"):
        ev.export_q_batch()
    ev.close()
    unbound = EmulEngine(rm, n_envs=2, q_cap=1024, bind=False)
    assert lib.sfl_export_q_batch(unbound.ctx, 0, 2, p(off), p(keys), p(vals), C.c_uint64(16), p(found), None) == -4
    assert b"sfl_bind first" in lib.sfl_last_error()
    unbound.close()
    # a table whose row count disagrees with its q_rows: more rows than counted are never written past the range
    counters = eng.buf["counters"].numpy()[:3 * backend.COUNTERS_DT.itemsize].view(backend.COUNTERS_DT)
    rows = counters["q_rows"].copy()
    for delta in (1, -1):
        counters["q_rows"][1] = rows[1] + delta
        with pytest.raises(RuntimeError, match="env 1: its Q table holds"):
            eng.export_q_batch()
    counters["q_rows"][1] = rows[1]
    assert eng.export_q_batch() == [eng.export_q(i) for i in range(3)]
    eng.close()


def c1_model(n_envs, default_q=0.0, engine=EmulSwitchEnv, fx=None):
    fx = fx if fx is not None else load_golden("c1_synth18")[0]
    rail_env = api.RailEnv(fx, malfunction_generator=api.ParamMalfunctionGen(api.MalfunctionParameters(0.01, 5, 15)))
    env = engine(rail_env, max_steps=100_000, n_envs=n_envs, q_cap=1024, ep_cap=2)
    return api.DistrQLearning(env=env, **HP, default_q=default_q, seed=450565)


def npz(path):
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


def assert_same_files(a_dir, b_dir, names):
    for name in names:
        if name.endswith(".pkl"):
            assert open(os.path.join(a_dir, name), "rb").read() == open(os.path.join(b_dir, name), "rb").read(), name
        else:
            za, zb = npz(os.path.join(a_dir, name)), npz(os.path.join(b_dir, name))
            assert list(za) == list(zb) == ["x"], name
            assert za["x"].dtype == zb["x"].dtype and np.array_equal(za["x"], zb["x"]), name


def checkpoint_names(n):
    return [f"checkpoint_{n}.pkl"] + [f"{k}_checkpoint_{n}.npz" for k in CKPT_NPZ]


def test_every_learner_gets_its_checkpoints():
    """learn(6 episodes, checkpoint_freq=3, exploit_freq=2) with ep_cap 2: the checkpoint before episode 2 comes between two
    launches and after an exploit rollout.  Every environment's checkpoint_3.pkl is the table of a same-seed learn() that
    stops there; its npz files have the primary environment's layout; out_dir is what it is without env_out_dirs."""
    dq = np.array([0.0, 0.5, 0.25])
    with tempfile.TemporaryDirectory() as tmp:
        dirs = [os.path.join(tmp, f"env_{i}") for i in range(3)]
        m = c1_model(3, dq)
        with pytest.raises(ValueError, match="2 directories for 3 environments"):
            m.learn(6, None, 3, 2, env_out_dirs=dirs[:2])
        m.learn(6, os.path.join(tmp, "out"), 3, 2, env_out_dirs=dirs)
        plain = c1_model(3, dq)
        plain.learn(6, os.path.join(tmp, "plain"), 3, 2)
        assert_same_files(os.path.join(tmp, "out"), os.path.join(tmp, "plain"), checkpoint_names(3) + checkpoint_names(6))
        assert sorted(os.listdir(os.path.join(tmp, "plain"))) == sorted(os.listdir(os.path.join(tmp, "out")))
        stopped = c1_model(3, dq)
        stopped.learn(2, None, 0, 2)
        for i, d in enumerate(dirs):
            assert sorted(os.listdir(d)) == sorted(checkpoint_names(3) + checkpoint_names(6))
            want = stopped.env.engine.export_q(i, include_init=True, default_q=float(dq[i]))
            assert open(os.path.join(d, "checkpoint_3.pkl"), "rb").read() == pkl_bytes(want), i
            assert api.read_q_table(os.path.join(d, "checkpoint_3.pkl")) == want
            mt = m.metrics
            for n, cut in ((3, 2), (6, 5)):
                z = {k: npz(os.path.join(d, f"{k}_checkpoint_{n}.npz")) for k in CKPT_NPZ}
                assert all(list(v) == ["x"] for v in z.values())
                assert np.array_equal(z["cum_reward"]["x"], np.concatenate([mt["cum_reward"][i, :cut], np.zeros(6 - cut)]))
                assert np.array_equal(z["arrived_trains"]["x"], mt["arrived_trains"][i, :cut])
                assert np.array_equal(z["delays"]["x"], mt["delays"][i, :cut])
                assert np.array_equal(z["num_malfunctions"]["x"], mt["num_malfunctions"][i, :cut])
                assert z["trains_at_dest"]["x"].shape == (0,)
            if i == m.primary_env:
                assert_same_files(d, os.path.join(tmp, "out"), checkpoint_names(3) + checkpoint_names(6))


def test_overlapped_writer_equals_writing_at_every_checkpoint_and_reraises():
    with tempfile.TemporaryDirectory() as tmp:
        runs = {}
        for overlap in (True, False):
            m = c1_model(2)
            m._overlap_checkpoints = overlap
            dirs = [os.path.join(tmp, f"{overlap}_{i}") for i in range(2)]
            m.learn(6, None, 2, None, env_out_dirs=dirs)
            runs[overlap] = dirs
        for a, b in zip(runs[True], runs[False]):
            assert_same_files(a, b, checkpoint_names(2) + checkpoint_names(4) + checkpoint_names(6))
        # a file the writer cannot create: learn() re-raises the writer's error in its own thread
        os.makedirs(os.path.join(tmp, "d1", "checkpoint_2.pkl"))
        m = c1_model(2)
        with pytest.raises(IsADirectoryError):
            m.learn(4, None, 2, None, env_out_dirs=[os.path.join(tmp, "d0"), os.path.join(tmp, "d1")])


def test_grid_writes_every_experiments_checkpoints_and_eval_reads_them():
    env_section = {"width": 18, "height": 18, "max_num_cities": 5, "max_rails_between_cities": 1, "max_rail_pairs_in_city": 1,
                   "number_of_agents": 2, "malfunction_rate": 0.05, "min_duration": 2, "max_duration": 5}
    hp = {"epsilon": [0.5, 0.1], "epsilon_decay_rate": [0.9997], "lr": [0.1], "lr_decay_rate": [1.0]}
    with tempfile.TemporaryDirectory() as tmp:
        dirs = cli.launch_grid(hp, random_seeds=[64, 65], out_dir=tmp, env_section=env_section, num_episodes=4, checkpoint_freq=2,
                               exploit_freq=None, env_cls=EmulSwitchEnv)
        assert len(dirs) == 4
        for d in dirs:
            for n in (2, 4):
                for name in checkpoint_names(n):
                    assert os.path.exists(os.path.join(d, name)), (d, name)
            with np.load(os.path.join(d, "delays_checkpoint_2.npz")) as z:
                assert z["x"].shape == (1, 2)
        res = cli.launch_eval(dirs, distr_q_model_name="checkpoint_2.pkl", env_cls=EmulSwitchEnv)
        assert set(res) == set(dirs) and all(r.shape == (2, 10) for r in res.values())
        # the final tables, through the batched export, are what save() of each environment's export_q writes
        fx = cli.fixture_from_env_section({k: str(v) for k, v in env_section.items()}, 64)
        env = EmulSwitchEnv(api.RailEnv(fx, malfunction_generator=api.ParamMalfunctionGen(api.MalfunctionParameters(0.05, 2, 5))),
                            max_steps=100_000, n_envs=2)
        m = api.DistrQLearning(env, gamma=1.0, epsilon=np.array([0.5, 0.1]), epsilon_decay_rate=np.array([0.9997] * 2),
                               lr=np.array([0.1] * 2), lr_decay_rate=np.array([1.0] * 2), default_q=0.0, seeds=[64, 64])
        m.learn(4, None, 0, None)
        for idx in range(2):
            want = pkl_bytes(env.engine.export_q(idx, include_init=True, default_q=0.0))
            assert open(os.path.join(tmp, f"exp_{idx}", "seed_0", "distr_q_model.pkl"), "rb").read() == want, idx


# ------------------------------------------------------------------------------------------------ on the B200
@pytest.mark.gpu
def test_cuda_compaction_at_c4_scale_equals_the_single_export():
    fx, _ = load_golden("c4_rail100_t50")
    rm = backend.RailMap(fx)
    n = 8192
    eng = backend.Engine(rm, n_envs=n, q_cap=65536, ep_cap=4)
    eng.set_hparams(**HP, default_q=0.0, seeds=np.arange(n) + 450565, episodes=-1)
    eng.reset()
    eng.enable_q_init(True)
    for _ in range(2):
        eng.run(backend.MODE_LEARN, 512)
    rows = eng.counters()["q_rows"]
    assert (rows > 0).all()
    snap = eng.compact_q(0, n)
    snap.wait()                                                           # every environment's count against q_rows
    assert int(snap.off[-1]) == int(rows.sum())
    for i in np.linspace(0, n - 1, 24).astype(int).tolist():
        keys, vals = snap.rows(i)
        want_k, want_v = eng.q_rows(i)
        assert np.array_equal(keys, want_k) and np.array_equal(vals, want_v), i
    sub = eng.export_q_batch(range(4000, 4003), include_init=True, default_q=0.0)
    assert sub == [eng.export_q(i, include_init=True, default_q=0.0) for i in range(4000, 4003)]
    eng.close()


@pytest.mark.gpu
def test_cuda_checkpoints_of_a_c3_grid_equal_the_host_build():
    """learn(env_out_dirs) on the C3 map, on the device (overlapped writer and writing at every checkpoint) and on the host
    build: the same pickles, byte for byte, and the same npz arrays."""
    fx, _ = load_golden("c3_synth80_s64")
    names = checkpoint_names(2) + checkpoint_names(4)
    with tempfile.TemporaryDirectory() as tmp:
        runs = {}
        for tag, engine, overlap in (("cuda", api.ASyncSwitchEnv, True), ("cuda_sync", api.ASyncSwitchEnv, False),
                                     ("host", EmulSwitchEnv, True)):
            rail_env = api.RailEnv(fx)
            env = engine(rail_env, max_steps=100_000, n_envs=6, q_cap=32768, ep_cap=2)
            m = api.DistrQLearning(env=env, **{**HP, "epsilon": np.linspace(0.2, 0.6, 6)}, default_q=0.0, seed=64)
            m._overlap_checkpoints = overlap
            runs[tag] = [os.path.join(tmp, tag, f"exp_{i}") for i in range(6)]
            m.learn(5, None, 2, 3, env_out_dirs=runs[tag])
            env.engine.close()
        for other in ("cuda_sync", "host"):
            for a, b in zip(runs["cuda"], runs[other]):
                assert_same_files(a, b, names)


def test_writer_drops_pending_checkpoints_when_learn_raises():
    """An exception in learn()'s own thread (an error, KeyboardInterrupt) ends the writer after the job it is running: the
    checkpoints still queued are not written before the exception surfaces."""
    ran = []
    with pytest.raises(KeyboardInterrupt):
        with api._CheckpointWriter(True) as w:
            started = threading.Event()
            w.submit(lambda: (started.set(), time.sleep(0.5), ran.append(1)), w.staging())
            w.submit(lambda: ran.append(2), w.staging())
            started.wait(5)
            raise KeyboardInterrupt
    assert ran == [1]
