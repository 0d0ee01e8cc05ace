"""Deterministic synthetic rail maps + timetables (SURVEY.md section 7 step 0, section 8f row N2).

flatland's ``sparse_rail_generator`` / ``sparse_line_generator`` (main.py:36-49) cannot be reproduced
without the upstream source, so benchmark and test maps come from this generator instead.  It only
emits the four switch shapes the reference supports (switch_agents.py:262-267), on square grids
(rail_graph.py:43-48 breaks non-square ones), with no dead ends, and keeps every (cell, heading) a
train can occupy connected to every cell:

  * start from one rectangular loop; a loop has a clockwise and a counter-clockwise "world" and a train
    never changes world because flatland trains cannot reverse;
  * repeatedly add a straight chord between two straight track cells.  In the clockwise world the chord
    is a one-way shortcut P -> Q (diverging simple switch at P, merging simple switch at Q; tracks it
    crosses become diamond crossings); the counter-clockwise world gets the mirror Q -> P.  Adding a
    path between two nodes of a strongly connected digraph keeps it strongly connected, so both worlds
    stay strongly connected and both cover every track cell.

The timetable restates flatland_patch/timetable_generators.py:23-136 on the greedy shortest paths.

A *fixture* is a plain dict: grid uint16[H,W], init_pos int32[T,2], init_dir int32[T], target int32[T,2],
earliest_departure int32[T], latest_arrival int32[T], max_episode_steps, malfunction_rate,
min_duration, max_duration, name.  ``save_fixture`` / ``load_fixture`` map it to one ``.npz``.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import numpy as np

from .railmap import DC, DR, INF_DIST, distance_to, shortest_path, trans_bit


def _bit(h: int, e: int) -> int:
    return 1 << (15 - (4 * h + e))


def _opp(d: int) -> int:
    return (d + 2) % 4


class _Builder:
    def __init__(self, n: int):
        self.n = n
        self.grid = np.zeros((n, n), np.int64)
        # clockwise-world heading per axis for straight track cells: axis 0 = vertical (N/S), 1 = horizontal (E/W)
        self.cw: Dict[Tuple[int, int], Dict[int, int]] = {}
        self.kind: Dict[Tuple[int, int], str] = {}     # 'straight' | 'curve' | 'switch' | 'cross'

    def _add(self, r, c, h, e):
        self.grid[r, c] |= _bit(h, e)

    def straight(self, r, c, heading):
        """bidirectional straight track; ``heading`` = clockwise-world heading on it."""
        self._add(r, c, heading, heading)
        self._add(r, c, _opp(heading), _opp(heading))
        self.cw.setdefault((r, c), {})[heading % 2 == 1 and 1 or 0] = heading
        self.kind[(r, c)] = "cross" if (r, c) in self.kind else "straight"

    def curve(self, r, c, h_in, h_out):
        """clockwise world turns h_in -> h_out; the other world turns opp(h_out) -> opp(h_in)."""
        self._add(r, c, h_in, h_out)
        self._add(r, c, _opp(h_out), _opp(h_in))
        self.kind[(r, c)] = "curve"

    def loop(self, r0, c0, r1, c1, reverse=False):
        """rectangular loop; the clockwise world runs it clockwise -- or counter-clockwise when ``reverse``."""
        if not reverse:
            for c in range(c0 + 1, c1):
                self.straight(r0, c, 1)      # top row heading E
                self.straight(r1, c, 3)      # bottom row heading W
            for r in range(r0 + 1, r1):
                self.straight(r, c1, 2)      # right column heading S
                self.straight(r, c0, 0)      # left column heading N
            self.curve(r0, c0, 0, 1)
            self.curve(r0, c1, 1, 2)
            self.curve(r1, c1, 2, 3)
            self.curve(r1, c0, 3, 0)
        else:
            for c in range(c0 + 1, c1):
                self.straight(r0, c, 3)
                self.straight(r1, c, 1)
            for r in range(r0 + 1, r1):
                self.straight(r, c1, 0)
                self.straight(r, c0, 2)
            self.curve(r0, c0, 3, 2)
            self.curve(r0, c1, 0, 3)
            self.curve(r1, c1, 1, 0)
            self.curve(r1, c0, 2, 1)

    def try_chord(self, p: Tuple[int, int], q: Tuple[int, int], rng) -> bool:
        """straight chord between p and q (same row or same column, at least one cell between)."""
        (pr, pc), (qr, qc) = p, q
        if pr == qr:
            axis, d = 1, (1 if qc > pc else 3)
            length = abs(qc - pc)
        elif pc == qc:
            axis, d = 0, (2 if qr > pr else 0)
            length = abs(qr - pr)
        else:
            return False
        if length < 2:
            return False
        for end in (p, q):
            if self.kind.get(end) != "straight" or (1 - axis) not in self.cw[end]:
                return False
        inner = [(pr + DR[d] * k, pc + DC[d] * k) for k in range(1, length)]
        for cell in inner:
            k = self.kind.get(cell)
            if k is None:
                continue
            if k == "straight" and (1 - axis) in self.cw[cell]:
                continue            # perpendicular straight -> diamond crossing
            return False
        # keep switches from touching each other along the track they sit on (neighbouring switches are
        # legal for the reference but rare in flatland maps; allow them only through crossings)
        for end in (p, q):
            for dd in range(4):
                nb = (end[0] + DR[dd], end[1] + DC[dd])
                if self.kind.get(nb) in ("switch",):
                    return False
        hp = self.cw[p][1 - axis]
        hq = self.cw[q][1 - axis]
        # clockwise world: p --d--> q
        self._add(pr, pc, hp, d)
        self._add(pr, pc, _opp(d), _opp(hp))
        self._add(qr, qc, d, hq)
        self._add(qr, qc, _opp(hq), _opp(d))
        self.kind[p] = "switch"
        self.kind[q] = "switch"
        for cell in inner:
            self.straight(cell[0], cell[1], d)
        return True


def generate_grid(n: int, n_chords: int, seed: int, margin: int = 1, allow_crossings: bool = True,
                  p_slip: float = 0.0) -> np.ndarray:
    """``p_slip``: probability that a diamond crossing becomes a single slip (Switch3, 7 actions) or, half of
    the time, a double slip (Switch4, 9 actions).  A slip lets the clockwise world turn from one track
    onto the other in that track's clockwise direction (and mirrors it for the other world)."""
    rng = np.random.RandomState(seed)
    b = _Builder(n)
    b.loop(margin, margin, n - 1 - margin, n - 1 - margin)
    added, tries = 0, 0
    while added < n_chords and tries < 200 * max(n_chords, 1):
        tries += 1
        straight = [cell for cell, k in b.kind.items() if k == "straight"]
        p = straight[rng.randint(len(straight))]
        axis = 1 - next(iter(b.cw[p]))        # chord runs perpendicular to p's track
        d = (0, 2)[rng.randint(2)] if axis == 0 else (1, 3)[rng.randint(2)]
        # walk from p in direction d until the first track cell that can terminate the chord
        r, c = p[0] + DR[d], p[1] + DC[d]
        q = None
        steps = 0
        while 0 <= r < n and 0 <= c < n:
            k = b.kind.get((r, c))
            steps += 1
            if k == "straight" and (1 - axis) in b.cw[(r, c)] and steps >= 2:
                if allow_crossings and rng.rand() < 0.35:
                    r, c = r + DR[d], c + DC[d]
                    continue          # cross it and keep going
                q = (r, c)
                break
            if k is not None and not (k == "straight" and (1 - axis) in b.cw[(r, c)]):
                break
            r, c = r + DR[d], c + DC[d]
        if q is None:
            continue
        ends = (p, q) if rng.rand() < 0.5 else (q, p)
        if b.try_chord(ends[0], ends[1], rng):
            added += 1
    if p_slip > 0:
        for cell in sorted(c for c, k in b.kind.items() if k == "cross"):
            if rng.rand() >= p_slip:
                continue
            hv, hh = b.cw[cell][0], b.cw[cell][1]
            first = (hh, hv) if rng.rand() < 0.5 else (hv, hh)
            pairs = [first] if rng.rand() < 0.5 else [first, (first[1], first[0])]
            for (a, z) in pairs:
                b._add(cell[0], cell[1], a, z)
                b._add(cell[0], cell[1], _opp(z), _opp(a))
    return b.grid.astype(np.uint16)


def generate_grid_v2(n: int, seed: int, n_rings: int = 2, ring_gap: int = 2, cross_every: int = 14, n_lines: int = 6,
                     double_lines: bool = True, p_slip: float = 0.2, margin: int = 1, with_headings: bool = False):
    """Double-track layout (stand-in for flatland's sparse_rail_generator with max_rails_between_cities = 2,
    hyperparam_tuning.py:17-26): ``n_rings`` concentric main-line loops ``ring_gap`` cells apart, joined by crossovers
    roughly every ``cross_every`` cells in alternating orientation, and ``n_lines`` interior lines across the innermost
    ring -- each a PAIR of parallel tracks two cells apart when ``double_lines`` -- so that opposing trains can pass
    each other instead of meeting head-on on a single track.  Built from the same two primitives as ``generate_grid``
    (loop + straight chord), so the strong-connectivity argument of the module docstring carries over: every ring is
    strongly connected in both worlds, and a chord only adds a path between two nodes of a strongly connected digraph
    (crossovers are added in both orientations between every pair of neighbouring rings).

    Right-hand running: in the clockwise world neighbouring rings run in OPPOSITE senses and the two tracks of a line
    pair in opposite directions, so that world alone reaches every place in both directions of travel on separate
    tracks -- a double-track railway under its normal operating rule.  ``with_headings`` also returns int8[n, n], the
    clockwise-world heading on every plain straight cell (-1 elsewhere), for ``make_fixture(headings=...)``: trains
    started with those headings all follow the rule; trains started against them run wrong-way and meet the others
    head-on, as on the single-track maps of ``generate_grid``."""
    rng = np.random.RandomState(seed)
    b = _Builder(n)
    rings = []
    for k in range(n_rings):
        m = margin + ring_gap * k
        if n - 1 - m - m < 6:
            break
        b.loop(m, m, n - 1 - m, n - 1 - m, reverse=bool(k % 2))
        rings.append(m)
    # ---- crossovers between neighbouring rings (alternating orientation, on all four sides)
    for k in range(len(rings) - 1):
        mo, mi = rings[k], rings[k + 1]
        lo, hi = mi + 2, n - 1 - mi - 2                       # keep clear of the corners of the inner ring
        flip = k % 2
        for side in range(4):
            pos = lo + int(rng.randint(0, max(cross_every // 2, 1)))
            while pos <= hi:
                if side == 0: p, q = (mo, pos), (mi, pos)                          # top
                elif side == 1: p, q = (pos, n - 1 - mo), (pos, n - 1 - mi)        # right
                elif side == 2: p, q = (n - 1 - mo, pos), (n - 1 - mi, pos)        # bottom
                else: p, q = (pos, mo), (pos, mi)                                  # left
                ends = (p, q) if flip else (q, p)
                if b.try_chord(ends[0], ends[1], rng):
                    flip ^= 1
                    pos += max(3, cross_every + int(rng.randint(-cross_every // 4, cross_every // 4 + 1)))
                else:
                    pos += 1
    # ---- interior lines across the innermost ring
    mi = rings[-1]
    added, tries = 0, 0
    while added < n_lines and tries < 400 * max(n_lines, 1):
        tries += 1
        vertical = bool(rng.randint(2))
        pos = int(rng.randint(mi + 3, n - 1 - mi - 4))
        if vertical: p, q, off = (mi, pos), (n - 1 - mi, pos), (0, 2)
        else: p, q, off = (pos, mi), (pos, n - 1 - mi), (2, 0)
        if rng.rand() < 0.5:
            p, q = q, p
        # a line may stop at the first earlier line it meets instead of crossing everything
        if rng.rand() < 0.5:
            d = (2 if q[0] > p[0] else 0) if vertical else (1 if q[1] > p[1] else 3)
            r, c = p[0] + DR[d], p[1] + DC[d]
            steps = 1
            while (r, c) != q:
                k_ = b.kind.get((r, c))
                axis = 0 if vertical else 1
                if k_ == "straight" and (1 - axis) in b.cw[(r, c)] and steps >= 4 and rng.rand() < 0.4:
                    q = (r, c)
                    break
                r, c = r + DR[d], c + DC[d]
                steps += 1
        p2, q2 = (p[0] + off[0], p[1] + off[1]), (q[0] + off[0], q[1] + off[1])
        snap = (b.grid.copy(), {k_: dict(v) for k_, v in b.cw.items()}, dict(b.kind))
        if not b.try_chord(p, q, rng):
            continue
        if double_lines and not b.try_chord(q2, p2, rng):      # the second track of the pair runs the other way
            b.grid, b.cw, b.kind = snap                      # keep lines double: undo the first track
            continue
        added += 1
    if p_slip > 0:
        for cell in sorted(c for c, k in b.kind.items() if k == "cross"):
            if rng.rand() >= p_slip:
                continue
            hv, hh = b.cw[cell][0], b.cw[cell][1]
            first = (hh, hv) if rng.rand() < 0.5 else (hv, hh)
            pairs = [first] if rng.rand() < 0.5 else [first, (first[1], first[0])]
            for (a, z) in pairs:
                b._add(cell[0], cell[1], a, z)
                b._add(cell[0], cell[1], _opp(z), _opp(a))
    grid = b.grid.astype(np.uint16)
    if not with_headings:
        return grid
    heads = np.full((n, n), -1, np.int8)
    for (r, c), k in b.kind.items():
        if k == "straight":
            heads[r, c] = next(iter(b.cw[(r, c)].values()))
    return grid, heads


def plain_cells(grid: np.ndarray) -> List[Tuple[int, int, int, int]]:
    """(r, c, heading_a, heading_b) for straight, non-crossing, non-switch track cells."""
    out = []
    H, W = grid.shape
    for r in range(H):
        for c in range(W):
            v = int(grid[r, c])
            if v == _bit(0, 0) | _bit(2, 2):
                out.append((r, c, 0, 2))
            elif v == _bit(1, 1) | _bit(3, 3):
                out.append((r, c, 1, 3))
    return out


def make_fixture(n: int = 18, n_trains: int = 2, n_chords: int = 4, seed: int = 0, num_cities: int = 2,
                 malfunction_rate: float = 0.0, min_duration: int = 0, max_duration: int = 0,
                 name: Optional[str] = None, p_slip: float = 0.0, grid: Optional[np.ndarray] = None, slack: float = 1.0,
                 headings: Optional[np.ndarray] = None, wrong_way: float = 0.0) -> dict:
    """``grid``: a ready transition grid (e.g. ``generate_grid_v2``) instead of the loop + chords generator;
    ``slack`` stretches the episode length and the arrival windows of the timetable; ``headings`` (from
    ``generate_grid_v2(with_headings=True)``): start every train with the right-hand-running heading of its cell, except
    a fraction ``wrong_way`` started against it."""
    if grid is None:
        grid = generate_grid(n, n_chords, seed, p_slip=p_slip)
    rng = np.random.RandomState(seed + 7919)
    cells = plain_cells(grid)
    # keep starts/targets away from switches so that _init_ports always walks at least one cell
    def near_switch(r, c):
        for d in range(4):
            rr, cc = r + DR[d], c + DC[d]
            if 0 <= rr < n and 0 <= cc < n and bin(int(grid[rr, cc])).count("1") > 2:
                return True
        return False
    cells = [x for x in cells if not near_switch(x[0], x[1])]
    if len(cells) < 2 * n_trains:
        raise ValueError("map too small for the requested number of trains")
    order = rng.permutation(len(cells))
    starts = [cells[i] for i in order[:n_trains]]
    tgts = [cells[i] for i in order[n_trains:2 * n_trains]]
    trains = []
    for (sr, sc, ha, hb), (tr, tc, _, _) in zip(starts, tgts):
        d0 = int((ha, hb)[rng.randint(2)])
        if headings is not None and headings[sr, sc] >= 0:
            d0 = int(headings[sr, sc])
            if rng.rand() < wrong_way:
                d0 = _opp(d0)
        trains.append(((sr, sc), d0, (tr, tc)))
    trains.sort(key=lambda t: t[0] + (t[1],))          # switch_env.py:104-119 ordering
    # ---- timetable (flatland_patch/timetable_generators.py:23-136, speed 1.0, single-leg lines)
    lens = []
    for (pos, d, tgt) in trains:
        dist = distance_to(grid, tgt)
        if dist[pos[0], pos[1], d] >= INF_DIST:
            raise ValueError("generator bug: unreachable target")
        lens.append(len(shortest_path(grid, dist, pos, d, tgt)))
    times = np.array(lens, dtype=float)
    max_steps_old = int(4 * 2 * (n + n + (n_trains / num_cities)))
    mean_delay = float(np.mean(times)) * 0.2
    max_steps_new = int(np.ceil(float(np.max(times)) * 1.5) + mean_delay)
    max_episode_steps = int(min(max_steps_new, int(max_steps_old * 3.0)) * slack)
    end_buffer = int(max_episode_steps * 0.05)
    la_max = max_episode_steps - end_buffer
    eds, las = [], []
    for t in times:
        travel_max = int(np.ceil(t * 1.3 + mean_delay))
        window = max(la_max - travel_max, 1)
        ed = int(rng.randint(0, window))
        eds.append(ed)
        las.append(ed + travel_max)
    return {
        "name": name or f"synth{n}x{n}_t{n_trains}_c{n_chords}_s{seed}",
        "grid": grid,
        "init_pos": np.array([t[0] for t in trains], np.int32),
        "init_dir": np.array([t[1] for t in trains], np.int32),
        "target": np.array([t[2] for t in trains], np.int32),
        "earliest_departure": np.array(eds, np.int32),
        "latest_arrival": np.array(las, np.int32),
        "max_episode_steps": int(max_episode_steps),
        "malfunction_rate": float(malfunction_rate),
        "min_duration": int(min_duration),
        "max_duration": int(max_duration),
    }


def loop_chord_fixture() -> dict:
    """The hand-built 7x7 'loop + chord' map of SURVEY.md Appendix C (KAT-1/KAT-2) with two trains."""
    g = np.zeros((7, 7), np.int64)
    def cell(r, c, pairs):
        for h, e in pairs:
            g[r, c] |= _bit(h, e)
    N, E, S, W = 0, 1, 2, 3
    cell(1, 1, [(N, E), (W, S)]); cell(1, 5, [(E, S), (N, W)]); cell(3, 5, [(E, N), (S, W)]); cell(3, 1, [(W, N), (S, E)])
    for rc in ((1, 2), (1, 4), (3, 2), (3, 4)):
        cell(*rc, [(E, E), (W, W)])
    for rc in ((2, 1), (2, 5), (2, 3)):
        cell(*rc, [(N, N), (S, S)])
    cell(1, 3, [(E, E), (E, S), (W, W), (N, W)])
    cell(3, 3, [(E, E), (E, N), (W, W), (S, W)])
    return {
        "name": "loop_chord_7x7",
        "grid": g.astype(np.uint16),
        "init_pos": np.array([[2, 1], [2, 5]], np.int32),
        "init_dir": np.array([0, 2], np.int32),       # both clockwise
        "target": np.array([[3, 4], [1, 2]], np.int32),
        "earliest_departure": np.array([0, 3], np.int32),
        "latest_arrival": np.array([14, 20], np.int32),
        "max_episode_steps": 60,
        "malfunction_rate": 0.0, "min_duration": 0, "max_duration": 0,
    }


def rail_fixture(n: int, n_trains: int, seed: int, n_rings: int = 2, n_lines: int = 8, cross_every: int = 10, p_slip: float = 0.2,
                 num_cities: int = 25, malfunction_rate: float = 0.0, min_duration: int = 0, max_duration: int = 0,
                 wrong_way: float = 0.0, name: Optional[str] = None) -> dict:
    """A double-track map (``generate_grid_v2``) with a right-hand-running timetable: the stand-in for flatland's
    ``sparse_rail_generator(max_rails_between_cities=2)`` + ``sparse_line_generator`` (main.py:36-49,
    hyperparam_tuning.py:17-26) that the C3 / C4 benchmark configurations and their goldens use."""
    grid, heads = generate_grid_v2(n, seed, n_rings=n_rings, n_lines=n_lines, cross_every=cross_every, p_slip=p_slip, with_headings=True)
    return make_fixture(n, n_trains, 0, seed=seed, num_cities=num_cities, malfunction_rate=malfunction_rate, min_duration=min_duration,
                        max_duration=max_duration, name=name or f"rail{n}_t{n_trains}_s{seed}", grid=grid, headings=heads,
                        wrong_way=wrong_way)


def c3_fixture(seed: int) -> dict:
    """BASELINE.json configs[2]: hyperparam_tuning.py:10-35 -- 80x80, 15 trains, 25 cities, rails 2/2, no malfunctions."""
    return rail_fixture(80, 15, seed, n_rings=2, n_lines=8, cross_every=10, num_cities=25, name=f"c3_rail80_s{seed}")


def c4_fixture() -> dict:
    """BASELINE.json configs[3]: large synthetic map -- 100x100, 50 trains, hundreds of switches, malfunctions 0.01 / 5-15."""
    return rail_fixture(100, 50, 0, n_rings=3, n_lines=20, cross_every=8, num_cities=25, malfunction_rate=0.01, min_duration=5,
                        max_duration=15, name="c4_rail100_t50")


def t100_fixture() -> dict:
    """The reference's 100-train evaluation (plot.ipynb "100_agents_challenge") on the C4 rail network: the map of
    ``c4_fixture`` with 100 trains on its timetable.  Generated from its seed, never stored."""
    return rail_fixture(100, 100, 0, n_rings=3, n_lines=20, cross_every=8, num_cities=25, malfunction_rate=0.01, min_duration=5,
                        max_duration=15, name="rail100_t100")


def offmap_malfunction_fixture() -> dict:
    """The 7x7 loop + chord map with two trains that share their entry cell (opposite headings): with injected
    malfunctions it exercises flatland's MALFUNCTION_OFF_MAP -> STOPPED transition onto an occupied cell (row F4)."""
    fx = loop_chord_fixture()
    fx.update(name="f4_offmap_7x7", init_pos=np.array([[2, 1], [2, 1]], np.int32), init_dir=np.array([0, 2], np.int32),
              target=np.array([[3, 4], [1, 2]], np.int32), earliest_departure=np.array([0, 2], np.int32),
              latest_arrival=np.array([30, 40], np.int32), max_episode_steps=80)
    return fx


_SCALARS = ("max_episode_steps", "malfunction_rate", "min_duration", "max_duration")


def save_fixture(path: str, fx: dict) -> None:
    np.savez_compressed(path, name=np.array(fx["name"]), **{k: np.asarray(v) for k, v in fx.items() if k != "name"})


def load_fixture(path: str) -> dict:
    with np.load(path, allow_pickle=False) as z:
        fx = {k: z[k] for k in z.files}
    fx["name"] = str(fx["name"])
    for k in _SCALARS:
        fx[k] = fx[k].item()
    return fx


def check_fixture(fx: dict) -> None:
    """Fail early on maps the reference cannot handle (see railmap.build_* for the cited checks)."""
    from .railmap import build_switch_tables, build_train_tables
    tab = build_switch_tables(fx["grid"])
    build_train_tables(tab, fx["init_pos"], fx["init_dir"], fx["target"], fx["earliest_departure"], fx["latest_arrival"])
