"""extend_semaphores (rail_network.py:229-244) through the trains' stop stamps.

A train that ends a tick STOPPED or MALFUNCTION slides the windows of the semaphore records it holds to start at that tick.
The kernels keep that tick in the train's TrB.stop_tick (SFL_NO_STOP before its first stop of the episode) and every reader
of a window start takes the later of the record's t0 and its holder's stamp (t0_eff).  The stamps live in the staged train
records, so they must survive launch boundaries and must not survive an episode reset.  These tests free-run learn() on
the reference's stream on congested golden maps, cut into launches of 1 and 7 ticks and into one launch for every episode,
and compare every decision and every present semaphore window (traced with t0_eff applied) with the reference's run; with
1-tick launches every stamp is also read back after every tick and compared with the one the reference's train states
imply.  On the GPU the same runs go through the full kernel, and the C4 learn kernel, cut the same ways, must equal the
host build."""
from __future__ import annotations

import numpy as np
import pytest

from switchfl_b200 import backend
from tests._parity import golden_events
from tests._util import hparams, load_golden
from tests.emulated import EmulEngine, build_emul
from tests.test_reference_stream import check_golden_free_run

NO_STOP = -2 ** 31
ST_STOPPED, ST_MALF = 4, 5
CONGESTED = ("synth40_t12", "c4_synth100_t50")          # the first has two episodes: its stamps cross a reset


def gpu_engine(rm, **kw):
    return backend.Engine(rm, device="cuda:0", **kw)


def stop_stamps(eng, env):
    """TrB.stop_tick of every train: the last word of each 16-byte TrB record.  An env block starts with the 248-byte header,
    word 1 of its train sets when T > 64, the reference stream's 48-byte state (at rng_offset, when there is one), then
    TrA[T] and TrB[T], 16-byte aligned (DESIGN.md section 3)."""
    T = eng.map.trains.T
    rng = int(eng.sizes.rng_offset)
    off = ((rng + 48 if rng else 248 + (32 if T > 64 else 0)) + 15) // 16 * 16 + 16 * T + int(eng.sizes.env_stride) * env
    raw = eng.buf["state"][off:off + 16 * T].cpu().numpy()
    return raw.view(np.int32).reshape(T, 4)[:, 3].copy()


def expected_stamps(g, i):
    """The stamps after logged tick i of the reference's run: per train, the last tick of that episode up to tick i at which
    the train's state was STOPPED or MALFUNCTION."""
    ep, tick, state = g["tick_ep"], g["tick_tick"], g["tick_state"]
    same = np.flatnonzero(ep[:i + 1] == ep[i])
    stopped = (state[same] == ST_STOPPED) | (state[same] == ST_MALF)
    last = np.where(stopped.any(0), (stopped.shape[0] - 1) - np.argmax(stopped[::-1], 0), -1)
    return np.where(last >= 0, tick[same][np.maximum(last, 0)], NO_STOP)


def check_stamps_tick_by_tick(name, factory, n_envs=2, lanes=None):
    fx, g = load_golden(name)
    rm = backend.RailMap(fx)
    n_dec, n_tick, n_ep = len(g["dec_action"]), len(g["tick_ep"]), int(g["n_episodes"])
    ev = golden_events(g)
    kw = {} if lanes is None else dict(lanes=lanes)
    eng = factory(rm, n_envs=n_envs, q_cap=1 << max(6, int(np.ceil(np.log2(len(g["q_keys"]) * 2 + 16)))), dec_cap=n_dec + 4,
                  tick_cap=n_tick + 4, ep_cap=n_ep + 1, ev_cap=len(ev) + 2, rng="reference", **kw)
    eng.set_hparams(**hparams(g), seeds=np.full(n_envs, int(g["seed"])), episodes=n_ep)
    eng.set_replay(None, [ev] * n_envs)
    eng.reset()
    eng.enable_q_init(True)
    n_stops = 0
    for _ in range(n_tick):
        eng.run(backend.MODE_LEARN, 1)
        c = eng.counters()
        i = int(c["n_tick_logged"][0]) - 1
        want = expected_stamps(g, i)
        n_stops += int((want != NO_STOP).sum())
        for env in range(n_envs):
            assert c["n_tick_logged"][env] == i + 1 and c["elapsed"][env] == g["tick_tick"][i], (name, env, i)
            assert np.array_equal(stop_stamps(eng, env), want), (name, env, i, stop_stamps(eng, env), want)
    eng.run(backend.MODE_LEARN, 8)
    c = eng.counters()
    assert (c["err"] == 0).all() and (c["halted"] == 1).all() and (c["decisions"] == n_dec).all(), c
    assert n_stops > 0
    eng.close()


@pytest.mark.parametrize("name", CONGESTED)
def test_emul_stamps_after_every_tick_equal_the_references_stops(name):
    build_emul()
    check_stamps_tick_by_tick(name, EmulEngine)


@pytest.mark.parametrize("chunk", (1, 7, "episode"))
@pytest.mark.parametrize("name", CONGESTED)
def test_emul_free_learn_cut_into_launches_equals_the_reference(name, chunk):
    build_emul()
    check_golden_free_run(name, EmulEngine, chunk=episode_chunk(name) if chunk == "episode" else chunk)


def episode_chunk(name):
    """Launches of one episode each: the longest episode of the reference's run, in ticks."""
    _, g = load_golden(name)
    return int(np.bincount(g["tick_ep"]).max())


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", CONGESTED)
def test_gpu_stamps_after_every_tick_equal_the_references_stops(name):
    for lanes in (8, 32):
        check_stamps_tick_by_tick(name, gpu_engine, lanes=lanes)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CONGESTED)
def test_gpu_free_learn_cut_into_launches_equals_the_reference(name):
    for chunk, lanes in ((1, 32), (7, 8), (episode_chunk(name), 32)):
        check_golden_free_run(name, gpu_engine, lanes=lanes, chunk=chunk)


HP_C4 = dict(gamma=0.95, epsilon=0.5, epsilon_decay_rate=0.999, lr=0.2, lr_decay_rate=1.0, default_q=1.0)


def c4_learn(cls, chunk, full=False, B=8, n_ep=2, **kw):
    """Free-running learn on the C4 map in launches of `chunk` ticks; everything observable, the stamps included."""
    fx, _ = load_golden("c4_rail100_t50")
    eng = cls(backend.RailMap(fx), n_envs=B, q_cap=32768, ep_cap=n_ep + 1, dec_cap=4 if full else 0, trace_sem=full, **kw)
    kernel = eng.kernel_variant(backend.MODE_LEARN, traced=full)
    eng.set_hparams(**HP_C4, seeds=np.arange(B) + 450565, episodes=n_ep)
    eng.reset()
    eng.enable_q_init(True)
    while not (eng.counters()["halted"] == 1).all():
        eng.run(backend.MODE_LEARN, chunk)
    eng.check_errors()
    c = eng.counters().copy()
    _, log, delays = eng.episode_log()
    out = ({k: c[k] for k in ("decisions", "ticks", "train_ticks", "episodes", "q_rows", "forced_stops", "stop_actions")},
           log[:, :n_ep].copy(), delays[:, :n_ep].copy(), [eng.export_q(i) for i in range(B)],
           [stop_stamps(eng, i) for i in range(B)])
    eng.close()
    return out, kernel


def assert_same(a, b):
    for k in a[0]:
        assert np.array_equal(a[0][k], b[0][k]), k
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and a[3] == b[3]
    assert all(np.array_equal(x, y) for x, y in zip(a[4], b[4]))


@pytest.mark.gpu
def test_gpu_c4_learn_and_full_kernels_cut_into_launches_equal_the_host_build():
    host, _ = c4_learn(EmulEngine, 1_000_000)
    for chunk, full in ((1, False), (7, False), (700, False), (7, True)):
        dev, kernel = c4_learn(gpu_engine, chunk, full=full, lanes=32, roomy=False)      # bench.py's C4 learn kernel
        assert kernel == "k_run<G=32,KIND=%s,TH=0,SQ=0,ONE=0,ROOMY=0>" % ("full" if full else "learn"), kernel
        assert_same(dev, host)
