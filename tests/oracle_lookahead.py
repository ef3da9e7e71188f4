"""Host restatement of the one-step lookahead map (cgl_env_action_rewards), for the tests.

rewards[a] = the reward of `toggle_state(a); step(); reward()` from the current planes, a = size the no-op.  On a torus
of side >= 3 a toggle at c changes only c and the neighbour count of its 8 neighbours, so

    R(c) = R_noop + H(c) + sum_{x in N8(c)} G_{d(c)}(x)        (mod 2^32),  d(c) = +1 if c is dead, -1 if alive

with G+-(x) = s'_x(count_x +- 1) - s'_x(count_x) and H(c) = s'_c(state flipped, stability set by the toggle) - s'_c.
Here every term is formed from the step rule itself (not from the closed forms the kernel uses), and sides 1 and 2,
where the torus aliases neighbours, are stepped by definition with the oracle.
"""
from __future__ import annotations

import numpy as np

from oracle import oracle


def _i8(x):
    return (np.asarray(x, np.int64) + 128) % 256 - 128


def next_stability(rule, s, alive, n, spawn, stable_max, empty, empty_min):
    """The stability after the step of cells with stability s, state alive and n live neighbours (int64 arrays)."""
    nxt = (n == 3) | ((n == 2) & alive)
    inc = np.where(s != stable_max, _i8(s + 1), s)
    if rule == oracle.DEAD_DECAY:
        dead = np.where(s != empty_min, _i8(s - 1), s)
    elif rule == oracle.DEAD_SAT:
        dead = np.minimum(_i8(s + empty), empty_min)
    else:
        dead = np.zeros_like(s)
    return np.where(nxt & alive, inc, np.where(nxt, spawn, dead))


def brute_force(world, stable, side, spawn, stable_max, rule=0, empty=0, empty_min=-128, masked=False):
    """Every action by definition: oracle toggle, step_rule, reward.  int32 [size + 1]."""
    size = side * side
    out = np.empty(size + 1, np.int32)
    for a in range(size + 1):
        w, s = world.copy(), stable.copy()
        if a < size:
            (oracle.toggle_masked if masked else oracle.toggle)(w, s, a, spawn)
        oracle.step_rule(w, s, side, spawn, stable_max, rule, empty, empty_min)
        out[a] = oracle.reward(s)
    return out


def action_rewards(world, stable, side, spawn, stable_max, rule=0, empty=0, empty_min=-128, masked=False, offset=0):
    """int32 [size + 1] for one env (world uint8 [size], stable int8 [size]).  `offset` is added to R_noop mod 2^32
    (what a plane near the int32 wrap of the sum would do to every entry)."""
    if side <= 2:
        out = brute_force(world, stable, side, spawn, stable_max, rule, empty, empty_min, masked)
        return ((out.astype(np.int64) + offset) % (1 << 32)).astype(np.uint32).view(np.int32)
    wb = world.reshape(side, side) != 0
    s = stable.reshape(side, side).astype(np.int64)
    n = sum(np.roll(np.roll(wb, dy, 0), dx, 1).astype(np.int64)
            for dy in (-1, 0, 1) for dx in (-1, 0, 1) if dy or dx)
    args = (spawn, stable_max, empty, empty_min)
    plain = next_stability(rule, s, wb, n, *args)
    gp = next_stability(rule, s, wb, n + 1, *args) - plain
    gm = next_stability(rule, s, wb, n - 1, *args) - plain
    put = np.where(masked & wb, 0, spawn)                  # the toggled cell is dead afterwards where it was alive
    h = next_stability(rule, put, ~wb, n, *args) - plain

    def box(p):
        return sum(np.roll(np.roll(p, dy, 0), dx, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if dy or dx)

    r_noop = int(plain.sum()) + offset
    delta = h + np.where(wb, box(gm), box(gp))
    full = np.append((r_noop + delta).reshape(-1), r_noop)
    return (full % (1 << 32)).astype(np.uint32).view(np.int32)


def batch(worlds, stables, side, spawn, stable_max, rule=0, empty=0, empty_min=-128, masked=False):
    """int32 [B, size + 1] for uint8 [B, size] worlds and int8 [B, size] planes."""
    return np.stack([action_rewards(w, s, side, spawn, stable_max, rule, empty, empty_min, masked)
                     for w, s in zip(worlds, stables)])
