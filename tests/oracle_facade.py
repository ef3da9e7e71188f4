"""Test helper: the `CGL.sim` facades' semantics on the C oracle, and the parameter corners of the single-env tests.

OracleEnv is what the base facade (`CGL.py`) and the fork's facade (`CGL_action+/CGL.py`) promise, restated on
`oracle.step_rule` / `oracle.toggle` / `oracle.toggle_masked` / `oracle.reward` / `oracle.alive`, with the lookahead
map of `oracle_lookahead` and the cycle stop of `oracle_cycle`.  tests/test_oracle_facade_cpu.py replays the golden
traces of the reference and of the fork through it, so the GPU tests that compare against it stand on the same
ground as the rest of the suite.
"""
from __future__ import annotations

import numpy as np

import oracle_cycle
import oracle_lookahead
from oracle import oracle

# (spawn, stable_max, dead_rule, empty, empty_min, masked).  The base rule at the reference's usual factors, at the
# int8 extremes and with spawn above max; the fork's two dead-cell rules at four (empty, empty_min) pairs, masked and
# unmasked; one masked base-rule corner.  23 corners: prime, so `side % len(CORNERS)` pairs every corner with every
# side % 4 class.
BASE_FACTORS = [(-2, 2), (-1, -1), (-128, 127), (127, -128), (0, 0), (5, 2)]
BASE_CORNERS = [(s, m, oracle.DEAD_ZERO, 0, -128, False) for s, m in BASE_FACTORS]
EMPTY_PAIRS = [(-1, -6), (127, -128), (-128, 127), (3, -3)]
FORK_CORNERS = [(*BASE_FACTORS[(2 * i + j + k) % len(BASE_FACTORS)], rule, e, emin, bool(k))
                for i, rule in enumerate((oracle.DEAD_DECAY, oracle.DEAD_SAT))
                for j, (e, emin) in enumerate(EMPTY_PAIRS) for k in (0, 1)]
CORNERS = BASE_CORNERS + FORK_CORNERS + [(-3, 4, oracle.DEAD_ZERO, 0, -128, True)]


def corner_plane(rs, size, corner):
    """An arbitrary int8 stability plane (dead cells included) in which about a third of the cells hold a value at or
    next to one of the corner's constants, so that every boundary of the rule is met even on small sides."""
    spawn, smax, _, empty, emin, _ = corner
    st = rs.randint(-128, 128, size=size).astype(np.int8)
    special = np.array([smax, smax - 1, smax + 1, smax & 0x7f, spawn, emin, emin + 1, emin - 1, empty, 0, 127, -128,
                        -1], np.int64)
    pick = rs.rand(size) < 0.35
    st[pick] = ((special[rs.randint(special.size, size=int(pick.sum()))] + 128) % 256 - 128).astype(np.int8)
    return st


class OracleEnv:
    """One env with the facade's methods, stepped by the C oracle.  fork=True: the fork's facade (dead cells follow
    `dead_rule`, start at `empty`, masked toggle, `load` carries `empty`, `update_state` may set the plane)."""

    def __init__(self, world, stable, side, spawn, stable_max, dead_rule=oracle.DEAD_ZERO, empty=0, empty_min=-128,
                 masked=False, fork=False):
        self.world = np.ascontiguousarray(world, np.uint8).reshape(-1).copy()
        self.stable = np.ascontiguousarray(stable, np.int8).reshape(-1).copy()
        self.side, self.size = side, side * side
        assert self.world.size == self.size == self.stable.size
        self.spawn, self.stable_max = spawn, stable_max
        self.dead_rule, self.empty, self.empty_min, self.masked, self.fork = dead_rule, empty, empty_min, masked, fork
        self.count = 0
        self._init = (self.world.copy(), self.stable.copy())

    @classmethod
    def seeded(cls, side, seed, spawn, stable_max, dead_rule=oracle.DEAD_ZERO, empty=0, empty_min=-128, masked=False,
               fork=False):
        """The facade's seeded start: the reference's random world, stability from spawn (and `empty`)."""
        world = oracle.initial_world(side, seed)
        return cls(world, oracle.initial_stable_fork(world, spawn, empty), side, spawn, stable_max, dead_rule, empty,
                   empty_min, masked, fork)

    # ---- the facade's methods
    def toggle_state(self, indx):
        (oracle.toggle_masked if self.masked else oracle.toggle)(self.world, self.stable, indx, self.spawn)

    def step(self):
        self.count += 1
        oracle.step_rule(self.world, self.stable, self.side, self.spawn, self.stable_max, self.dead_rule, self.empty,
                         self.empty_min)

    def run(self, iters, until_fixed=False):
        n = oracle.run_rule(self.world, self.stable, self.side, self.spawn, self.stable_max, iters, self.dead_rule,
                            self.empty, self.empty_min, until_fixed=until_fixed)
        self.count += n
        return n

    def run_until_cycle(self, iters, max_period=2):
        n, p = oracle_cycle.run_cycle(self.world, self.stable, self.side, self.spawn, self.stable_max, iters, max_period,
                                      self.dead_rule, self.empty, self.empty_min)
        self.count += n
        return n, p

    def reward(self):
        return int(oracle.reward(self.stable))

    def alive(self):
        return int(oracle.alive(self.world))

    def action_rewards(self):
        return oracle_lookahead.action_rewards(self.world, self.stable, self.side, self.spawn, self.stable_max,
                                               self.dead_rule, self.empty, self.empty_min, self.masked)

    def reset(self):
        """Back to the start of this side (count untouched): the seeded start, or what a load that changed the side
        brought (its world, stability initialised from spawn and `empty`)."""
        self.world, self.stable = self._init[0].copy(), self._init[1].copy()

    def match(self, cells):
        return bool(np.array_equal(self.world, np.asarray(cells).reshape(-1)))

    def update_state(self, world, stable=None):
        self.world = np.ascontiguousarray(world, np.uint8).reshape(-1).copy()
        if stable is not None:
            self.stable = np.ascontiguousarray(stable, np.int8).reshape(-1).copy()

    def save(self):
        out = (self.world.copy(), self.stable.copy(), self.side, self.count, self.spawn, self.stable_max)
        return out + (self.empty,) if self.fork else out

    def load(self, world, stable, side, count, spawn, stable_max, empty=None):
        if self.fork:
            self.empty = empty
        resized = side != self.side
        self.side, self.size, self.count, self.spawn, self.stable_max = side, side * side, count, spawn, stable_max
        self.world = np.ascontiguousarray(world, np.uint8).reshape(-1).copy()
        self.stable = np.ascontiguousarray(stable, np.int8).reshape(-1).copy()
        if resized:
            self._init = (self.world.copy(), oracle.initial_stable_fork(self.world, spawn, self.empty))
