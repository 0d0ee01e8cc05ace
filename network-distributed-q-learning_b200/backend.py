"""ctypes binding of the C-ABI (include/switchfl_b200.h) + the batched engine object the drop-in classes use.

PyTorch only owns the device buffers (one uint8 tensor per buffer of ``sfl_buffers``); every bit of the
hot path runs inside ``libswitchfl_b200.so`` (hand-written sm_100a CUDA).  There is no CPU fallback: if
the library is missing or no CUDA device exists, construction raises.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import railmap

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libswitchfl_b200.so")

ABI_VERSION = 10
MODE_LEARN, MODE_GREEDY, MODE_REPLAY, MODE_STEP = 0, 1, 2, 3
RNG_PHILOX, RNG_REFERENCE = 0, 1
RNG_NAMES = {"philox": RNG_PHILOX, "reference": RNG_REFERENCE}
MALF_PHILOX, MALF_REFERENCE = 0, 1
MALF_NAMES = {"philox": MALF_PHILOX, "reference": MALF_REFERENCE}
ERR_NO_TRAIN_AT_SWITCH = 1
ERR_BITS = {1: "no train at active switch (observer.py:294-307)", 2: "infinite distance to target (observer.py:35-36)",
            4: "per-env Q table full (raise q_cap)", 8: "pending-update list full (raise pend_cap)",
            16: "train action plan overflow", 32: "replay action stream exhausted", 64: "invalid action (switch_env.py:213-215)",
            128: "replay diverged: an action recorded as greedy is not the argmax of the Q row"}

_i32p, _u16p, _i8p, _u8p = C.POINTER(C.c_int32), C.POINTER(C.c_uint16), C.POINTER(C.c_int8), C.POINTER(C.c_uint8)


class MapDesc(C.Structure):
    _fields_ = [("H", C.c_int32), ("W", C.c_int32), ("S", C.c_int32), ("NP", C.c_int32), ("NA", C.c_int32), ("T", C.c_int32),
                ("NT", C.c_int32), ("max_episode_steps", C.c_int32), ("grid", _u16p), ("cell_switch", _i32p),
                ("sw_P", _i32p), ("sw_A", _i32p), ("sw_port0", _i32p), ("sw_act0", _i32p),
                ("port_nbr", _i32p), ("port_dist", _i32p), ("port_n_intra", _i32p), ("port_intra0", _i32p),
                ("act_in", _i32p), ("act_out", _i32p), ("act_move", _i32p),
                ("init_cell", _i32p), ("init_dir", _i32p), ("target_cell", _i32p), ("ed", _i32p), ("la", _i32p),
                ("first_port", _i32p), ("first_dist", _i32p), ("init_delay", _i32p), ("tgt_index", _i32p),
                ("dist", _i32p), ("qinit_act", _i8p), ("qinit_final", _u8p)]


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_envs", "q_cap", "pend_cap", "max_steps", "dec_cap", "tick_cap", "ep_cap",
                                         "act_cap", "ev_cap", "trace_sem", "shared_q", "rng", "malf_rng", "eval_q")]


class Sizes(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("state_bytes", "env_stride", "hparams_bytes", "trace_dec_bytes", "trace_tick_bytes",
                                          "trace_sem_bytes", "ep_log_bytes", "ep_delay_bytes", "replay_act_bytes",
                                          "replay_ev_bytes", "counters_bytes", "step_out_bytes", "shared_q_bytes", "shared_d_bytes",
                                          "shared_c_bytes")] + [("q_stride", C.c_int32), ("a_max", C.c_int32), ("rng_offset", C.c_uint64),
                                                                  ("eval_q_bytes", C.c_uint64)]


class Buffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("state", "hparams", "counters", "trace_dec", "trace_tick", "trace_sem", "ep_log",
                                          "ep_delay", "replay_act", "replay_ev", "step_out", "shared_q", "shared_d", "shared_c",
                                          "eval_q")]


HPARAMS_DT = np.dtype([("gamma", "f8"), ("epsilon", "f8"), ("epsilon_decay_rate", "f8"), ("lr", "f8"), ("lr_decay_rate", "f8"),
                       ("default_q", "f8"), ("seed", "u8"), ("malf_threshold", "u4"), ("malf_min", "i4"), ("malf_max", "i4"),
                       ("episodes", "i4"), ("episode_base", "i4"), ("malf_thr2", "u4")])
COUNTERS_DT = np.dtype([("decisions", "u8"), ("ticks", "u8"), ("train_ticks", "u8"), ("episodes", "i4"), ("err", "i4"),
                        ("q_rows", "i4"), ("halted", "i4"), ("n_dec_logged", "i4"), ("n_tick_logged", "i4"),
                        ("n_ep_logged", "i4"), ("elapsed", "i4"), ("aborted", "i4"), ("reserved", "i4"),
                        ("forced_stops", "u8"), ("stop_actions", "u8"), ("arrived_trains", "u8"), ("reserved2", "u8"),
                        ("phase_cycles", "u8", (6,))])
DEC_DT = np.dtype([("ep", "i4"), ("tick", "i4"), ("sw", "i4"), ("train", "i4"), ("key", "u4"), ("mask", "i4"), ("action", "i4"),
                   ("next_sw", "i4"), ("reward", "i4"), ("done", "i4"), ("arrived", "u8"), ("arrived_hi", "u8")])
TICK_DT = np.dtype([("pos", "i4"), ("dir", "i1"), ("state", "i1"), ("malf", "i2")])
STEP_DT = np.dtype([("pending", "i4"), ("sw", "i4"), ("train", "i4"), ("key", "u4"), ("mask", "i4"), ("done", "i4"), ("elapsed", "i4"),
                    ("last_next_sw", "i4"), ("arrived", "u8"), ("rewards", "i4", (128,)), ("arrived_hi", "u8")])
EP_DT = np.dtype([("cum_reward", "f8"), ("decisions", "i4"), ("arrived", "i4"), ("num_malfunctions", "i4"), ("ticks", "i4"), ("arrived_mask", "u8"),
                  ("arrived_mask_hi", "u8")])
assert HPARAMS_DT.itemsize == 80 and COUNTERS_DT.itemsize == 144 and DEC_DT.itemsize == 56 and TICK_DT.itemsize == 8 and EP_DT.itemsize == 40
assert STEP_DT.itemsize == 560


def train_set(lo, hi, T: int) -> List[int]:
    """The trains of a record's two-word train set (``arrived`` / ``arrived_hi``, ``arrived_mask`` / ``arrived_mask_hi``):
    bit t of ``lo`` is train t, bit t of ``hi`` is train 64 + t; ascending train handles."""
    lo, hi = int(lo), int(hi)
    return [h for h in range(T) if ((lo >> h) if h < 64 else (hi >> (h - 64))) & 1]


def load_library(path: Optional[str] = None) -> C.CDLL:
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(path)
    lib.sfl_last_error.restype = C.c_char_p
    lib.sfl_query_sizes.argtypes = [C.POINTER(MapDesc), C.POINTER(Config), C.POINTER(Sizes)]
    lib.sfl_create.argtypes = [C.POINTER(MapDesc), C.POINTER(Config), C.c_int, C.POINTER(C.c_void_p)]
    lib.sfl_destroy.argtypes = [C.c_void_p]
    lib.sfl_bind.argtypes = [C.c_void_p, C.POINTER(Buffers)]
    lib.sfl_reset.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.sfl_enable_q_init.argtypes = [C.c_void_p, C.c_int]
    lib.sfl_reapply_q_init.argtypes = [C.c_void_p, C.c_void_p]
    lib.sfl_set_lanes.argtypes = [C.c_void_p, C.c_int]
    lib.sfl_get_lanes.argtypes = [C.c_void_p]
    lib.sfl_set_cta_warps.argtypes = [C.c_void_p, C.c_int]
    lib.sfl_set_roomy.argtypes = [C.c_void_p, C.c_int]
    lib.sfl_set_phase_clock.argtypes = [C.c_void_p, C.c_int]
    lib.sfl_describe_launch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_int]
    lib.sfl_run.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.sfl_total_decisions.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p]
    lib.sfl_export_q.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_int), C.c_void_p]
    lib.sfl_import_q.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.c_int, C.c_void_p]
    lib.sfl_set_eval_table.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.c_int, C.c_void_p]
    lib.sfl_shared_q_apply.argtypes = [C.c_void_p, C.c_void_p]
    lib.sfl_shared_q_apply_to.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sfl_kat_q_update.argtypes = [C.POINTER(C.c_double), C.c_int32, C.POINTER(C.c_double), C.c_int]
    lib.sfl_kat_pcg64.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int32, C.c_int32, C.POINTER(C.c_uint64), C.c_int]
    lib.sfl_kat_explore.argtypes = [C.POINTER(C.c_double), C.c_int32, C.POINTER(C.c_int32), C.c_int]
    lib.sfl_malf_schedule.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_int32), C.c_void_p]
    lib.sfl_distance_map.argtypes = [_u16p, C.c_int32, C.c_int32, _i32p, C.c_int32, _i32p, C.c_int]
    if lib.sfl_abi_version() != ABI_VERSION:
        raise RuntimeError("switchfl_b200 ABI version mismatch")
    return lib


def device_distance_map(grid: np.ndarray, target_cells: Sequence[int], device: int = 0, lib: Optional[C.CDLL] = None) -> np.ndarray:
    """int32[NT, H, W, 4] distance map of flatland_patch/distance_map.py:62-167 computed on the GPU (``sfl_distance_map``);
    same values as the host BFS ``railmap.distance_to`` (which the goldens pin against the vendored reference code)."""
    lib = lib or load_library()
    g = np.ascontiguousarray(grid, np.uint16)
    tg = np.ascontiguousarray(target_cells, np.int32)
    H, W = g.shape
    out = np.empty((len(tg), H, W, 4), np.int32)
    rc = lib.sfl_distance_map(g.ctypes.data_as(_u16p), H, W, tg.ctypes.data_as(_i32p), len(tg), out.ctypes.data_as(_i32p), int(device))
    if rc != 0:
        raise RuntimeError(f"switchfl_b200 error {rc}: {lib.sfl_last_error().decode()}")
    return out


def device_q_update(rows: Sequence[Sequence[float]], device: int = 0, lib: Optional[C.CDLL] = None) -> np.ndarray:
    """``sfl_kat_q_update``: the device's Q-update arithmetic on rows of (q, lr, reward, gamma, max_next, bootstrap)."""
    lib = lib or load_library()
    a = np.ascontiguousarray(rows, np.float64).reshape(-1, 6)
    out = np.empty(len(a), np.float64)
    rc = lib.sfl_kat_q_update(a.ctypes.data_as(C.POINTER(C.c_double)), len(a), out.ctypes.data_as(C.POINTER(C.c_double)), int(device))
    if rc != 0:
        raise RuntimeError(f"switchfl_b200 error {rc}: {lib.sfl_last_error().decode()}")
    return out


def device_pcg64(gens, codes, device: int = 0, lib: Optional[C.CDLL] = None):
    """``sfl_kat_pcg64``: the device's copy of the reference's random stream (SFL_RNG_REFERENCE).  ``gens``: rows of
    (state_hi, state_lo, inc_hi, inc_lo, has_uint32, uinteger), or (0, seed, 0, 0, 0, 0) for ``np.random.default_rng(seed)``;
    ``codes[g]``: the draws of generator g (0: random(), 1..2^32: integers(0, code), 2^63 | mask: one exploring decision).
    Returns (states after seeding [n, 6], results [n, n_codes] as uint64, final states [n, 6])."""
    lib = lib or load_library()
    g = np.ascontiguousarray(np.asarray(gens, dtype=object).astype(np.uint64)).reshape(-1, 6)
    c = np.ascontiguousarray(np.asarray(codes, dtype=object).astype(np.uint64)).reshape(len(g), -1)
    out = np.zeros((len(g), 12 + c.shape[1]), np.uint64)
    u64p = C.POINTER(C.c_uint64)
    rc = lib.sfl_kat_pcg64(g.ctypes.data_as(u64p), c.ctypes.data_as(u64p), len(g), c.shape[1], out.ctypes.data_as(u64p), int(device))
    if rc != 0:
        raise RuntimeError(f"switchfl_b200 error {rc}: {lib.sfl_last_error().decode()}")
    return out[:, :6], out[:, 6:6 + c.shape[1]], out[:, 6 + c.shape[1]:]


def device_explore(rows, device: int = 0, lib: Optional[C.CDLL] = None) -> np.ndarray:
    """``sfl_kat_explore``: the kernel's epsilon test on rows of (u, epsilon, decay, n, running product of the decay)."""
    lib = lib or load_library()
    a = np.ascontiguousarray(rows, np.float64).reshape(-1, 5)
    out = np.zeros(len(a), np.int32)
    rc = lib.sfl_kat_explore(a.ctypes.data_as(C.POINTER(C.c_double)), len(a), out.ctypes.data_as(C.POINTER(C.c_int32)), int(device))
    if rc != 0:
        raise RuntimeError(f"switchfl_b200 error {rc}: {lib.sfl_last_error().decode()}")
    return out.astype(bool)


def pcg64_state(words) -> dict:
    """numpy's ``bit_generator.state`` of a PCG64 from the kernel's words (state_hi, state_lo, inc_hi, inc_lo, has_uint32, uinteger)."""
    w = [int(x) for x in words]
    return {"bit_generator": "PCG64", "state": {"state": (w[0] << 64) | w[1], "inc": (w[2] << 64) | w[3]},
            "has_uint32": w[4], "uinteger": w[5]}


def side_ok(engine) -> bool:
    """True on a CUDA engine (streams exist); the host build of the tests runs the overlapped schedule serially."""
    return engine.device.type == "cuda"


def malf_threshold(rate: float) -> int:
    """ParamMalfunctionGen probability 1 - exp(-rate) (SURVEY.md Appendix B) as a 32-bit threshold."""
    if rate <= 0:
        return 0
    return min(int((1.0 - math.exp(-rate)) * 4294967296.0), 0xFFFFFFFF)


def malf_prob(rate: float) -> float:
    """flatland's malfunction probability per (train, tick), computed as ParamMalfunctionGen.prob does."""
    return 0.0 if rate <= 0 else 1.0 - math.exp(-rate)


def malf_hit_below(rate: float) -> int:
    """ceil(p * 2^53) for p = malf_prob(rate): a draw rand() = k * 2^-53 hits iff the integer k is below it
    (SFL_MALF_REFERENCE)."""
    return math.ceil(malf_prob(rate) * 2.0 ** 53)


def reference_ev_cap(fixture: dict) -> int:
    """Events per environment that flatland's malfunction schedule of this map fits in: the mean of the binomial
    T * max_episode_steps draws plus a wide margin (16 standard deviations + 64), at most one per draw."""
    n = len(fixture["init_dir"]) * int(fixture["max_episode_steps"])
    p = malf_prob(float(fixture["malfunction_rate"]))
    return max(1, min(n, int(math.ceil(n * p + 16.0 * math.sqrt(n * p * (1.0 - p)))) + 64))


def malf_thr2(threshold: int) -> int:
    """Stage-2 threshold of the two-stage malfunction draw: floor(thr * 256 / B) with B = ceil(thr / 2^24)."""
    if threshold <= 0:
        return 0
    b = (threshold + 0xFFFFFF) >> 24
    return min((threshold << 8) // b, 0xFFFFFFFF)


class RailMap:
    """Everything derived from one fixture: port-graph tables, per-train constants, the C descriptor."""

    def __init__(self, fixture: dict, device_bfs: Optional[int] = None):
        """``device_bfs``: CUDA device index to compute the distance map with ``sfl_distance_map`` (None: host BFS)."""
        self.fixture = fixture
        self.tab = railmap.build_switch_tables(fixture["grid"])
        dist_fn = None if device_bfs is None else (lambda grid, cells: device_distance_map(grid, cells, device=device_bfs))
        self.trains = railmap.build_train_tables(self.tab, fixture["init_pos"], fixture["init_dir"], fixture["target"],
                                                 fixture["earliest_departure"], fixture["latest_arrival"], dist_fn=dist_fn)
        t, tr = self.tab, self.trains
        self._keep = {}

        def arr(name, a, dt=np.int32):
            a = np.ascontiguousarray(a, dtype=dt)
            self._keep[name] = a
            return a

        d = MapDesc()
        d.H, d.W, d.S, d.NP, d.NA, d.T, d.NT = t.H, t.W, t.S, t.NP, len(t.act_in), tr.T, len(tr.targets)
        d.max_episode_steps = int(fixture["max_episode_steps"])
        d.grid = arr("grid", t.grid, np.uint16).ctypes.data_as(_u16p)
        for name, a in (("cell_switch", t.cell_switch), ("sw_P", t.sw_P), ("sw_A", t.sw_A), ("sw_port0", t.sw_port0),
                        ("sw_act0", t.sw_act0), ("port_nbr", t.port_nbr), ("port_dist", t.port_dist),
                        ("port_n_intra", t.port_n_intra), ("port_intra0", t.port_intra0), ("act_in", t.act_in),
                        ("act_out", t.act_out), ("act_move", t.act_move), ("init_cell", tr.init_cell), ("init_dir", tr.init_dir),
                        ("target_cell", tr.target_cell), ("ed", tr.ed), ("la", tr.la), ("first_port", tr.first_port),
                        ("first_dist", tr.first_dist), ("init_delay", tr.init_delay), ("tgt_index", tr.tgt_index),
                        ("dist", tr.dist)):
            setattr(d, name, arr(name, a).ctypes.data_as(_i32p))
        d.qinit_act = arr("qinit_act", tr.qinit_act, np.int8).ctypes.data_as(_i8p)
        d.qinit_final = arr("qinit_final", (tr.qinit_val == 1000.0), np.uint8).ctypes.data_as(_u8p)
        self.desc = d

    # ---- state-index <-> observation (observer.py:303-306 layout [row, col, sem[P], target[2P], delay[P]])
    def key_to_obs(self, key: int) -> tuple:
        t, tr = self.tab, self.trains
        NT = len(tr.targets)
        port, rem = divmod(int(key), NT * 48)
        tgt, rem = divmod(rem, 48)
        semb, level = divmod(rem, 3)
        s = int(t.port_switch[port])
        P = int(t.sw_P[s])
        cur = port - int(t.sw_port0[s])
        r, c = t.switch_cells[s]
        tcell = int(tr.targets[tgt])
        sem = [(semb >> k) & 1 for k in range(P)]
        target = [-1] * (2 * P)
        target[2 * cur], target[2 * cur + 1] = tcell // t.W, tcell % t.W
        delay = [-1] * P
        delay[cur] = level
        return (int(r), int(c), *sem, *target, *delay)

    def obs_to_key(self, obs: Sequence[int]) -> int:
        t, tr = self.tab, self.trains
        s = t.switch_cells.index((int(obs[0]), int(obs[1])))
        P = int(t.sw_P[s])
        sem = obs[2:2 + P]
        target = obs[2 + P:2 + 3 * P]
        delay = obs[2 + 3 * P:2 + 4 * P]
        cur = [k for k in range(P) if delay[k] >= 0][0]
        tcell = int(target[2 * cur]) * t.W + int(target[2 * cur + 1])
        tgt = int(np.where(tr.targets == tcell)[0][0])
        semb = sum(int(sem[k]) << k for k in range(P))
        return (((int(t.sw_port0[s]) + cur) * len(tr.targets) + tgt) * 16 + semb) * 3 + int(delay[cur])

    def q_arrays(self, q: Dict[tuple, List[float]], a_max: int):
        """The reference's dict as (uint32[n] state keys, float64[n, a_max] values, zero-padded): ``obs_to_key`` of every
        observation, computed per group of equally long observations and rows with array operations."""
        t, tr = self.tab, self.trains
        NT = len(tr.targets)
        n = len(q)
        keys = np.zeros(max(n, 1), np.uint32)
        vals = np.zeros((max(n, 1), a_max), np.float64)
        if not n:
            return keys, vals
        # (row, col) -> switch and target cell -> target index: the first match, as list.index / np.where in obs_to_key
        cell_sw = np.full(t.H * t.W, -1, np.int64)
        for s in range(len(t.switch_cells) - 1, -1, -1):
            r, c = t.switch_cells[s]
            cell_sw[int(r) * t.W + int(c)] = s
        cell_tgt = np.full(t.H * t.W, -1, np.int64)
        targets = np.asarray(tr.targets, np.int64)
        cell_tgt[targets[::-1]] = np.arange(NT - 1, -1, -1)
        port0 = np.asarray(t.sw_port0, np.int64)
        groups: Dict[tuple, List[int]] = {}
        items = list(q.items())
        for i, (obs, row) in enumerate(items):
            groups.setdefault((len(obs), len(row)), []).append(i)
        for (lo, lr), idx in groups.items():
            P = (lo - 2) // 4
            idx = np.asarray(idx)
            o = np.array([items[i][0] for i in idx], np.int64).reshape(len(idx), lo)
            vals[idx, :lr] = np.array([items[i][1] for i in idx], np.float64).reshape(len(idx), lr)
            s = cell_sw[o[:, 0] * t.W + o[:, 1]]
            delay = o[:, 2 + 3 * P:2 + 4 * P]
            cur = np.argmax(delay >= 0, axis=1)
            rows = np.arange(len(idx))
            tgt = cell_tgt[o[rows, 2 + P + 2 * cur] * t.W + o[rows, 3 + P + 2 * cur]]
            if (s < 0).any() or (tgt < 0).any() or not (delay >= 0).any(axis=1).all():
                raise ValueError("an observation of the Q table is not one of this map's states")
            semb = (o[:, 2:2 + P] << np.arange(P)).sum(axis=1)
            keys[idx] = ((((port0[s] + cur) * NT + tgt) * 16 + semb) * 3 + delay[rows, cur]).astype(np.uint32)
        return keys, vals

    def q_init_rows(self, default_q: float) -> Dict[tuple, List[float]]:
        """All rows __init_q_table creates (distr_q.py:81-181), as the reference's dict."""
        t, tr = self.tab, self.trains
        out = {}
        NT = len(tr.targets)
        for port in range(t.NP):
            s = int(t.port_switch[port])
            P, A = int(t.sw_P[s]), int(t.sw_A[s])
            for tgt in range(NT):
                a = int(tr.qinit_act[port, tgt])
                if a < 0:
                    continue
                for semb in range(1, 1 << P):
                    for level in range(3):
                        row = [default_q] * A
                        row[a] = float(tr.qinit_val[port, tgt])
                        out[self.key_to_obs(((port * NT + tgt) * 16 + semb) * 3 + level)] = row
        return out


class Engine:
    """B lockstep environments of one map on one GPU: owns the torch buffers and the C context."""

    def __init__(self, rail_map: RailMap, n_envs: int, device: str = "cuda:0", q_cap: int = 1024, pend_cap: int = 8,
                 max_steps: int = 100_000, dec_cap: int = 0, tick_cap: int = 0, ep_cap: int = 64, act_cap: int = 0,
                 ev_cap: int = 0, trace_sem: bool = False, lanes: Optional[int] = None, shared_q: bool = False,
                 cta_warps: Optional[int] = None, roomy: Optional[bool] = None, phase_clock: bool = False, bind: bool = True,
                 rng: str = "philox", malfunction_rng: str = "philox", eval_q: bool = False):
        """``bind=False`` creates the context only (no device buffers): enough for ``describe_launch``.
        ``eval_q``: an evaluation context -- greedy runs only, every environment reading ONE read-only Q table of ``q_cap``
        rows (``set_eval_table``) instead of a private table; the environments keep no Q region.
        ``rng``: the epsilon-greedy stream of learn mode -- "philox" (the specialised learn kernels) or "reference" (numpy's
        PCG64 stream of the reference learner, seeded per environment from its seed at every reset that restarts the
        interaction counters: a seeded learn() makes the reference's decisions; runs on the full kernel).
        ``malfunction_rng``: "philox" (the counter-based draws) or "reference" (flatland's ``RandomState(seed)`` stream:
        every environment's malfunction schedule is generated on the device from its seed, rate and durations by
        ``reset()``, and applied in every mode; learn runs on the full kernel).  With "reference" and ``ev_cap=0`` the
        schedule's capacity is sized from the fixture (``reference_ev_cap``)."""
        if rng not in RNG_NAMES:
            raise ValueError(f"rng must be one of {sorted(RNG_NAMES)}, not {rng!r}")
        if malfunction_rng not in MALF_NAMES:
            raise ValueError(f"malfunction_rng must be one of {sorted(MALF_NAMES)}, not {malfunction_rng!r}")
        self.rng = rng
        self.malfunction_rng = malfunction_rng
        if malfunction_rng == "reference" and not ev_cap:
            ev_cap = reference_ev_cap(rail_map.fixture)
        import torch
        self.torch = torch
        self.map = rail_map
        self.n_envs = int(n_envs)
        self.lib, self.device, dev_index = self._open(device)
        self.cfg = Config(n_envs=self.n_envs, q_cap=q_cap, pend_cap=pend_cap, max_steps=max_steps, dec_cap=dec_cap,
                          tick_cap=tick_cap, ep_cap=ep_cap, act_cap=act_cap, ev_cap=ev_cap, trace_sem=int(trace_sem),
                          shared_q=int(shared_q), rng=RNG_NAMES[rng], malf_rng=MALF_NAMES[malfunction_rng], eval_q=int(eval_q))
        self.shared_q = bool(shared_q)
        self.eval_q = bool(eval_q)
        self.eval_rows = 0                                # rows of the evaluation table (set_eval_table)
        self.sizes = Sizes()
        self._ck(self.lib.sfl_query_sizes(C.byref(rail_map.desc), C.byref(self.cfg), C.byref(self.sizes)))
        self.ctx = C.c_void_p()
        self._ck(self.lib.sfl_create(C.byref(rail_map.desc), C.byref(self.cfg), dev_index, C.byref(self.ctx)))
        if lanes is not None:
            self._ck(self.lib.sfl_set_lanes(self.ctx, int(lanes)))
        if cta_warps is not None:
            self._ck(self.lib.sfl_set_cta_warps(self.ctx, int(cta_warps)))
        if roomy is not None:
            self._ck(self.lib.sfl_set_roomy(self.ctx, int(bool(roomy))))
        if phase_clock:
            self._ck(self.lib.sfl_set_phase_clock(self.ctx, 1))
        self.phase_clock = bool(phase_clock)
        self.hparams = np.zeros(self.n_envs, HPARAMS_DT)
        self.malfunction_rate = float(rail_map.fixture["malfunction_rate"])
        self._malf_key = None                             # (seeds, rate, min, max) of the generated schedules
        self.max_malfunction_events = 0                   # events of the longest generated schedule
        self._pinned = {}
        self._pinned_ev = {}
        self.buf = {}
        self.reset_io_counters()
        if not bind:
            return
        z = lambda n: torch.zeros(max(int(n), 16), dtype=torch.uint8, device=self.device)
        s = self.sizes
        self.buf = {"state": z(s.state_bytes), "hparams": z(s.hparams_bytes), "counters": z(s.counters_bytes),
                    "trace_dec": z(s.trace_dec_bytes), "trace_tick": z(s.trace_tick_bytes), "trace_sem": z(s.trace_sem_bytes),
                    "ep_log": z(s.ep_log_bytes), "ep_delay": z(s.ep_delay_bytes), "replay_act": z(s.replay_act_bytes),
                    "replay_ev": z(s.replay_ev_bytes), "step_out": z(s.step_out_bytes), "shared_q": z(s.shared_q_bytes),
                    "shared_d": z(s.shared_d_bytes), "shared_c": z(s.shared_c_bytes), "eval_q": z(s.eval_q_bytes)}
        b = Buffers(**{k: v.data_ptr() for k, v in self.buf.items()})
        self._ck(self.lib.sfl_bind(self.ctx, C.byref(b)))

    # ------------------------------------------------------------------ helpers
    def _open(self, device):
        """(library, torch device of the buffers, CUDA device index)."""
        torch = self.torch
        if not torch.cuda.is_available():
            raise RuntimeError("switchfl_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        dev = torch.device(device)
        return load_library(), dev, dev.index or 0

    @staticmethod
    def bfs_device(device) -> Optional[int]:
        """CUDA device index the map preprocessing (distance map) runs on."""
        import torch
        return torch.device(device).index or 0

    def _ck(self, rc: int):
        if rc != 0:
            raise RuntimeError(f"switchfl_b200 error {rc}: {self.lib.sfl_last_error().decode()}")

    def reset_io_counters(self):
        """Bytes copied host->device / device->host through this engine and kernel launches since the last call."""
        self.h2d_bytes = self.d2h_bytes = self.n_launches = 0

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _upload(self, name: str, host: np.ndarray):
        """host -> device through a reusable pinned staging buffer."""
        torch = self.torch
        raw = np.ascontiguousarray(host).view(np.uint8).reshape(-1)
        self.h2d_bytes += raw.size
        dst = self.buf[name][:raw.size]
        st = self._pinned.get(name)
        if st is None or st.numel() < raw.size:
            st = self._pinned[name] = torch.empty(raw.size, dtype=torch.uint8, pin_memory=True)
            self._pinned_ev[name] = torch.cuda.Event()
        else:
            self._pinned_ev[name].synchronize()            # the previous copy out of this staging buffer has finished
        st[:raw.size].copy_(torch.from_numpy(raw))
        dst.copy_(st[:raw.size], non_blocking=True)
        self._pinned_ev[name].record(torch.cuda.current_stream(self.device))

    def _download(self, name: str, nbytes: Optional[int] = None) -> np.ndarray:
        """device -> host; small buffers that are read every step (counters, step records) go through a reusable pinned
        staging buffer, everything else through a plain copy."""
        t = self.buf[name] if nbytes is None else self.buf[name][:nbytes]
        self.d2h_bytes += t.numel()
        if t.numel() > (8 << 20):
            return t.cpu().numpy()
        torch = self.torch
        st = self._pinned.get("d2h:" + name)
        if st is None or st.numel() < t.numel():
            st = self._pinned["d2h:" + name] = torch.empty(t.numel(), dtype=torch.uint8, pin_memory=True)
        st[:t.numel()].copy_(t, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return st[:t.numel()].numpy().copy()

    def close(self):
        if getattr(self, "ctx", None) is not None and self.ctx:
            self.lib.sfl_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ control
    def set_hparams(self, gamma=1.0, epsilon=0.4, epsilon_decay_rate=0.0, lr=0.4, lr_decay_rate=0.0, default_q=0.0,
                    seeds=None, episodes=-1, episode_base=0, malfunction_rate=None, min_duration=None, max_duration=None):
        """Scalars broadcast; arrays give one value per env (the hyper-parameter / seed grid)."""
        fx = self.map.fixture
        hp = self.hparams
        for k, v in (("gamma", gamma), ("epsilon", epsilon), ("epsilon_decay_rate", epsilon_decay_rate), ("lr", lr),
                     ("lr_decay_rate", lr_decay_rate), ("default_q", default_q), ("episodes", episodes),
                     ("episode_base", episode_base)):
            hp[k] = v
        hp["seed"] = np.arange(self.n_envs, dtype=np.uint64) if seeds is None else np.asarray(seeds, np.uint64)
        rate = fx["malfunction_rate"] if malfunction_rate is None else malfunction_rate
        self.malfunction_rate = float(rate)
        hp["malf_threshold"] = malf_threshold(float(rate))
        hp["malf_thr2"] = malf_thr2(int(hp["malf_threshold"][0]))
        hp["malf_min"] = fx["min_duration"] if min_duration is None else min_duration
        hp["malf_max"] = fx["max_duration"] if max_duration is None else max_duration
        self._upload("hparams", hp)

    def reset(self, keep_q: bool = False, keep_interactions: bool = False):
        """``malfunction_rng="reference"``: first (re)generates the malfunction schedules when the seeds, the rate or the
        durations changed since they were last generated -- every path (learn(), learn_chunk(), test(), the AEC reset)
        goes through here."""
        if self.malfunction_rng == "reference":
            self._malf_generate()
        self._ck(self.lib.sfl_reset(self.ctx, int(keep_q) | (int(keep_interactions) << 1), self._stream()))

    def _malf_generate(self):
        hp = self.hparams
        key = (hp["seed"].tobytes(), self.malfunction_rate, hp["malf_min"].tobytes(), hp["malf_max"].tobytes())
        if key == self._malf_key:
            return
        hit = np.full(self.n_envs, malf_hit_below(self.malfunction_rate), np.uint64)
        n = C.c_int32()
        self._malf_key = None
        rc = self.lib.sfl_malf_schedule(self.ctx, hit.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(n), self._stream())
        self.max_malfunction_events = n.value             # also when the schedules do not fit: the ev_cap they need
        self._ck(rc)
        self._malf_key = key

    def malfunction_schedule(self, env: int) -> np.ndarray:
        """``malfunction_rng="reference"``: environment ``env``'s schedule, int32 rows (tick, train, duration) in tick order --
        every malfunction flatland draws for ticks 1 .. max_episode_steps; one is applied when the train's counter is 0."""
        if self.malfunction_rng != "reference":
            raise RuntimeError('malfunction_schedule() needs Engine(malfunction_rng="reference")')
        self._malf_generate()
        cap = self.cfg.ev_cap
        ev = self.buf["replay_ev"][int(env) * cap * 12:(int(env) + 1) * cap * 12].cpu().numpy().view(np.int32).reshape(cap, 3)
        end = np.nonzero(ev[:, 0] < 0)[0]
        return ev[:int(end[0]) if len(end) else cap].copy()

    @property
    def lanes(self) -> int:
        """Lanes of a warp cooperating on one environment (a scheduling choice; results do not depend on it)."""
        return int(self.lib.sfl_get_lanes(self.ctx))

    def reapply_q_init(self):
        """Overwrite the existing rows of optimistic-init states with their initial values in every environment's table
        (``sfl_reapply_q_init``: what __init_q_table does to a non-empty table, distr_q.py:156-158, 179-181)."""
        self._ck(self.lib.sfl_reapply_q_init(self.ctx, self._stream()))

    def describe_launch(self, mode: int = MODE_LEARN, traced: bool = False) -> str:
        """The kernel instantiation + launch configuration ``run(mode)`` would use (``sfl_describe_launch``)."""
        buf = C.create_string_buffer(256)
        self._ck(self.lib.sfl_describe_launch(self.ctx, int(mode), int(traced), buf, 256))
        return buf.value.decode()

    def kernel_variant(self, mode: int = MODE_LEARN, traced: bool = False) -> str:
        return self.describe_launch(mode, traced).split(" ")[0]

    def enable_q_init(self, on: bool = True):
        self._ck(self.lib.sfl_enable_q_init(self.ctx, int(on)))

    def run(self, mode: int, max_ticks: int):
        self.n_launches += 1
        self._ck(self.lib.sfl_run(self.ctx, int(mode), int(max_ticks), self._stream()))

    def set_replay(self, actions: Optional[Sequence[Sequence[int]]], events: Optional[Sequence[np.ndarray]] = None):
        """actions[i]: the recorded action stream of env i; events[i]: int array [(tick, train, duration)].  With
        ``malfunction_rng="reference"`` the schedule comes from the seeds alone: ``events`` must be None."""
        if self.malfunction_rng == "reference" and events is not None:
            raise ValueError('set_replay(events=...) with malfunction_rng="reference": the schedule is generated from the seeds')
        if actions is not None:
            a = np.full((self.n_envs, self.cfg.act_cap), -1, np.int8)
            for i, s in enumerate(actions):
                a[i, :len(s)] = s
            self._upload("replay_act", a)
        if self.cfg.ev_cap and self.malfunction_rng != "reference":
            ev = np.full((self.n_envs, self.cfg.ev_cap, 3), -1, np.int32)
            for i, e in enumerate(events or []):
                e = np.asarray(e, np.int32).reshape(-1, 3)
                e = e[np.lexsort((e[:, 1], e[:, 0]))] if len(e) else e
                ev[i, :len(e)] = e
            self._upload("replay_ev", ev)

    # ------------------------------------------------------------------ shared-table mode (extension, DESIGN.md section 7)
    def _shared_cells(self) -> int:
        return self.map.tab.NP * len(self.map.trains.targets) * 48 * self.sizes.a_max

    def init_shared_q(self, default_q: float = 0.0, q_init: bool = True):
        """Fill the shared table: default_q everywhere, the optimistic rows of distr_q.py:81-181 when ``q_init``."""
        assert self.shared_q
        t, tr = self.map.tab, self.map.trains
        NT, a_max = len(tr.targets), self.sizes.a_max
        q = np.full((t.NP, NT, 16, 3, a_max), float(default_q), np.float64)
        if q_init:
            port, tgt = np.nonzero(np.asarray(tr.qinit_act) >= 0)
            act = np.asarray(tr.qinit_act)[port, tgt]
            val = np.asarray(tr.qinit_val)[port, tgt]
            for semb in range(1, 16):                                   # every semaphore vector except all-red (:98-125)
                q[port, tgt, semb, :, act] = val[:, None]
        self._upload("shared_q", q)
        self.buf["shared_d"].zero_()
        self.buf["shared_c"].zero_()
        sq = getattr(self, "_sq", None)
        if sq is not None:                                                # the second table / accumulator pair of run_shared
            sq["q"][1].copy_(sq["q"][0]); sq["d"][1].zero_(); sq["c"][1].zero_()
            sq["step"], sq["done"] = 0, [None, None]

    def shared_q_sync(self, dist=None):
        """Fold the accumulated TD steps into the table; with an initialised ``torch.distributed`` first sum the
        accumulators over all ranks (integer all-reduce: NCCL on the GPU box, gloo in the CPU tests)."""
        assert self.shared_q
        self._allreduce_accumulators(dist, self.buf["shared_d"], self.buf["shared_c"])
        self._ck(self.lib.sfl_shared_q_apply(self.ctx, self._stream()))

    def _allreduce_accumulators(self, dist, d_buf, c_buf):
        if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
            n = self._shared_cells()
            dist.all_reduce(d_buf[:n * 8].view(self.torch.int64), op=dist.ReduceOp.SUM)
            dist.all_reduce(c_buf[:n * 4].view(self.torch.int32), op=dist.ReduceOp.SUM)

    # Overlapped schedule: two tables and two accumulator pairs.  Step k reads table T_k = buf[k % 2] and accumulates into
    # pair k % 2; its synchronisation (all-reduce + apply) runs on a SECOND stream while the kernel of step k + 1 already
    # reads T_{k+1}, and produces T_{k+2} = T_{k+1} + mean step of pair k % 2 in the buffer T_k occupied.  The TD steps are
    # thus folded in one step late -- a fixed, deterministic delay (integer sums): the result does not depend on timing,
    # on the number of ranks or on whether anything actually overlapped (the host build runs the same schedule serially).
    def _sq_setup(self):
        if getattr(self, "_sq", None) is None:
            torch = self.torch
            z = lambda n: torch.zeros(max(int(n), 16), dtype=torch.uint8, device=self.device)
            s = self.sizes
            self._sq = {"q": [self.buf["shared_q"], z(s.shared_q_bytes)], "d": [self.buf["shared_d"], z(s.shared_d_bytes)],
                        "c": [self.buf["shared_c"], z(s.shared_c_bytes)], "step": 0, "done": [None, None], "side": self._side_stream()}
            self._sq["q"][1].copy_(self._sq["q"][0])                    # T_0 = T_1 = the initial table
        return self._sq

    def _side_stream(self):
        return self.torch.cuda.Stream(device=self.device)

    def _bind_shared(self, q, d, c):
        b = Buffers(**{k: v.data_ptr() for k, v in self.buf.items()})
        b.shared_q, b.shared_d, b.shared_c = q.data_ptr(), d.data_ptr(), c.data_ptr()
        self._ck(self.lib.sfl_bind(self.ctx, C.byref(b)))

    def run_shared(self, max_ticks: int, dist=None, mode: int = MODE_LEARN):
        """One step of shared-table learning on the overlapped schedule (call ``init_shared_q`` first)."""
        assert self.shared_q
        torch, sq = self.torch, self._sq_setup()
        k = sq["step"] % 2
        main, side = (torch.cuda.current_stream(self.device), sq["side"]) if side_ok(self) else (None, None)
        if main is not None and sq["done"][k] is not None:
            main.wait_event(sq["done"][k])                              # T_k is complete, pair k is cleared
        self._bind_shared(sq["q"][k], sq["d"][k], sq["c"][k])
        self.run(mode, max_ticks)
        if main is None:                                                # host build: the same schedule, serially
            self._allreduce_accumulators(dist, sq["d"][k], sq["c"][k])
            self._ck(self.lib.sfl_shared_q_apply_to(self.ctx, sq["q"][1 - k].data_ptr(), sq["q"][k].data_ptr(), sq["d"][k].data_ptr(),
                                                    sq["c"][k].data_ptr(), None))
        else:
            ran = torch.cuda.Event()
            ran.record(main)
            with torch.cuda.stream(side):
                side.wait_event(ran)
                self._allreduce_accumulators(dist, sq["d"][k], sq["c"][k])
                self._ck(self.lib.sfl_shared_q_apply_to(self.ctx, sq["q"][1 - k].data_ptr(), sq["q"][k].data_ptr(), sq["d"][k].data_ptr(),
                                                        sq["c"][k].data_ptr(), C.c_void_p(side.cuda_stream)))
                sq["done"][k] = torch.cuda.Event()
                sq["done"][k].record(side)
        sq["step"] += 1

    def shared_q_flush(self):
        """Wait for the outstanding synchronisations of ``run_shared`` and make the newest table the bound one."""
        sq = getattr(self, "_sq", None)
        if sq is None or sq["step"] == 0:
            return
        if side_ok(self):
            sq["side"].synchronize()
        newest = (sq["step"] - 1) % 2
        if newest != 0:                                                 # keep buf["shared_q"] the table the exporters read
            self.buf["shared_q"].copy_(sq["q"][1])
        else:
            sq["q"][1].copy_(sq["q"][0])
        sq["step"], sq["done"] = 0, [None, None]
        self._bind_shared(self.buf["shared_q"], self.buf["shared_d"], self.buf["shared_c"])

    def shared_q_table(self) -> np.ndarray:
        """The shared table as float64[NP, NT, 16 semaphore vectors, 3 delay levels, a_max]."""
        t, tr = self.map.tab, self.map.trains
        n = self._shared_cells()
        self.shared_q_flush()                                             # outstanding run_shared synchronisations
        return self._download("shared_q", n * 8).view(np.float64).reshape(t.NP, len(tr.targets), 16, 3, self.sizes.a_max).copy()

    def export_shared_q(self, default_q: float = 0.0) -> Dict[tuple, List[float]]:
        """Rows of the shared table that differ from ``default_q`` somewhere, in the reference's dict layout."""
        q = self.shared_q_table()
        t = self.map.tab
        out = {}
        for port, tgt, semb, level in zip(*np.nonzero((q != float(default_q)).any(axis=-1))):
            s_ = int(t.port_switch[port])
            if semb >> int(t.sw_P[s_]):
                continue                                                # bits beyond the switch's ports are never produced
            key = ((int(port) * q.shape[1] + int(tgt)) * 16 + int(semb)) * 3 + int(level)
            out[self.map.key_to_obs(key)] = [float(x) for x in q[port, tgt, semb, level, :int(t.sw_A[s_])]]
        return out

    # ------------------------------------------------------------------ host-driven AEC protocol (SFL_MODE_STEP)
    def step(self, actions: Optional[Sequence[int]] = None, max_ticks: Optional[int] = None) -> np.ndarray:
        """Apply ``actions[i]`` to the decision waiting in env i (ignored where none waits), advance every env to
        its next decision point and return the per-env ``sfl_step_rec`` array (what AECEnv.last() reports)."""
        if self.cfg.act_cap < 1:
            raise RuntimeError("Engine(act_cap >= 1) is needed for the step protocol")
        a = np.full((self.n_envs, self.cfg.act_cap), -1, np.int8)
        if actions is not None:
            a[:, 0] = np.asarray(actions, np.int64).reshape(self.n_envs)
        self._upload("replay_act", a)
        self.run(MODE_STEP, int(self.map.fixture["max_episode_steps"]) + 2 if max_ticks is None else max_ticks)
        return self._download("step_out", self.n_envs * STEP_DT.itemsize).view(STEP_DT).copy()

    # ------------------------------------------------------------------ results
    def rng_state(self, env: Optional[int] = None):
        """The reference stream's state of every environment (or of ``env``) in numpy's ``bit_generator.state`` layout:
        ``np.random.Generator(np.random.PCG64())`` with this state continues where the environment's learner stands."""
        if self.rng != "reference":
            raise RuntimeError('rng_state() needs Engine(rng="reference")')
        off, stride = int(self.sizes.rng_offset), int(self.sizes.env_stride)
        envs = range(self.n_envs) if env is None else [int(env)]
        out = []
        for i in envs:
            raw = self.buf["state"][i * stride + off:i * stride + off + 48].cpu().numpy()
            w = raw[:32].view(np.uint64)
            out.append(pcg64_state([w[0], w[1], w[2], w[3], *raw[32:40].view(np.uint32)]))
        return out if env is None else out[0]

    def total_decisions(self):
        d, t = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.sfl_total_decisions(self.ctx, C.byref(d), C.byref(t), self._stream()))
        return d.value, t.value

    def counters(self) -> np.ndarray:
        c = self._download("counters", self.n_envs * COUNTERS_DT.itemsize).view(COUNTERS_DT)
        return c

    def check_errors(self, allow: int = 0):
        """Raise on any per-env error bit not in ``allow`` (the reference raises / asserts at these points)."""
        err = self.counters()["err"] & ~np.int32(allow)
        if err.any():
            i = int(np.nonzero(err)[0][0])
            msgs = [m for b, m in ERR_BITS.items() if err[i] & b]
            raise RuntimeError(f"env {i}: {'; '.join(msgs)} ({int((err != 0).sum())} env(s) flagged)")

    def episode_log(self):
        n = self.counters()["n_ep_logged"]
        log = self._download("ep_log").view(EP_DT)[:self.n_envs * self.cfg.ep_cap].reshape(self.n_envs, self.cfg.ep_cap)
        T = self.map.trains.T
        delays = self._download("ep_delay").view(np.int32)[:self.n_envs * self.cfg.ep_cap * T].reshape(self.n_envs, self.cfg.ep_cap, T)
        return n, log, delays

    def trace(self, env: int):
        c = self.counters()[env]
        T, NP = self.map.trains.T, self.map.tab.NP
        dec = self._download("trace_dec", self.n_envs * self.cfg.dec_cap * DEC_DT.itemsize).view(DEC_DT).reshape(self.n_envs, self.cfg.dec_cap)[env]
        dec = dec[:min(int(c["n_dec_logged"]), self.cfg.dec_cap)]
        tick = self._download("trace_tick", self.n_envs * self.cfg.tick_cap * T * TICK_DT.itemsize).view(TICK_DT).reshape(self.n_envs, self.cfg.tick_cap, T)[env]
        tick = tick[:min(int(c["n_tick_logged"]), self.cfg.tick_cap)]
        sem = None
        if self.cfg.trace_sem:
            sem = self._download("trace_sem").view(np.int32)[:self.n_envs * self.cfg.dec_cap * NP * 4]
            sem = sem.reshape(self.n_envs, self.cfg.dec_cap, NP, 4)[env][:len(dec)]
        return dec, tick, sem

    def q_rows(self, env: int):
        """The rows of env ``env``'s Q hash table in slot order: (uint32[n] state keys, float64[n, a_max] values)."""
        a_max = self.sizes.a_max
        cap = self.cfg.q_cap
        keys = np.zeros(cap, np.uint32)
        vals = np.zeros((cap, a_max), np.float64)
        n = C.c_int()
        self._ck(self.lib.sfl_export_q(self.ctx, env, keys.ctypes.data_as(C.POINTER(C.c_uint32)),
                                       vals.ctypes.data_as(C.POINTER(C.c_double)), cap, C.byref(n), self._stream()))
        return keys[:n.value], vals[:n.value]

    def export_q(self, env: int, include_init: bool = False, default_q: Optional[float] = None) -> Dict[tuple, List[float]]:
        """The reference's q_table dict (distr_q.py:42, pickled by :521-523): obs tuple -> list of A floats."""
        if self.shared_q:
            return self.export_shared_q(float(self.hparams["default_q"][env]) if default_q is None else default_q)
        keys, vals = self.q_rows(env)
        out = {}
        if include_init:
            out.update(self.map.q_init_rows(float(self.hparams["default_q"][env]) if default_q is None else default_q))
        t = self.map.tab
        NT = len(self.map.trains.targets)
        for k, v in zip(keys, vals):
            A = int(t.sw_A[t.port_switch[int(k) // (NT * 48)]])
            out[self.map.key_to_obs(int(k))] = [float(x) for x in v[:A]]
        return out

    def import_q(self, env: int, q: Dict[tuple, List[float]]):
        keys, vals = self.map.q_arrays(q, self.sizes.a_max)
        self._ck(self.lib.sfl_import_q(self.ctx, env, keys.ctypes.data_as(C.POINTER(C.c_uint32)),
                                       vals.ctypes.data_as(C.POINTER(C.c_double)), len(q), self._stream()))

    def set_eval_table(self, q: Dict[tuple, List[float]]):
        """``eval_q``: fill the evaluation table with the reference's dict (observation tuple -> list of A floats), hashed on
        the host and uploaded once (``sfl_set_eval_table``).  Needs ``q_cap`` above the row count."""
        if not self.eval_q:
            raise RuntimeError("set_eval_table() needs Engine(eval_q=True)")
        keys, vals = self.map.q_arrays(q, self.sizes.a_max)
        self._ck(self.lib.sfl_set_eval_table(self.ctx, keys.ctypes.data_as(C.POINTER(C.c_uint32)),
                                             vals.ctypes.data_as(C.POINTER(C.c_double)), len(q), self._stream()))
        self.h2d_bytes += int(self.sizes.eval_q_bytes)
        self.eval_rows = len(q)
