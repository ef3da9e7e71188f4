"""CPU suite: env runs that stop at the first repeated world of any period (cgl_env_run_settle).

The host restatement of the device's finder, tests/oracle_settle.py, is checked against a brute force that remembers
every past world (tests/oracle_cycle.py:run_cycle with max_period = max_steps), on thousands of random small tori with
budgets around each board's mu + lambda.  That pins the checkpoint schedule and the 2M bound independently of the
GPU.  The argument checks of cgl_env_run_settle run before any device work."""
import ctypes

import numpy as np
import pytest

from oracle import oracle
from oracle_cycle import run_cycle
from oracle_settle import checkpoint, find_settle, run_settle

GLIDER = [(0, 1), (1, 2), (2, 0), (2, 1), (2, 2)]
LWSS = [(0, 1), (0, 4), (1, 0), (2, 0), (2, 4), (3, 0), (3, 1), (3, 2), (3, 3)]         # 2*side on even sides, 4*side on odd ones


def place(side, cells, r0=2, c0=2):
    w = np.zeros(side * side, dtype=np.uint8)
    for r, c in cells:
        w[((r0 + r) % side) * side + (c0 + c) % side] = 1
    return w


def brute_force(world, side, max_steps, stable=None, args=(-2, 3, 0, 0, -128)):
    """(t, p) with every past world kept; the world (and stable, if given) are stepped in place."""
    s = np.zeros(world.size, np.int8) if stable is None else stable
    spawn, smax, rule, empty, emin = args
    return run_cycle(world, s, side, spawn, smax, max_steps, max(max_steps, 1), rule, empty, emin)


def _settle_time(w, side, limit=5000):
    """mu + lambda of the world, or None past `limit`."""
    t, p = brute_force(w.copy(), side, limit)
    return t if p else None


def test_checkpoint_schedule():
    assert [t for t in range(40) if checkpoint(t, 20)] == [0, 1, 2, 4, 8, 16, 20]
    assert [t for t in range(40) if checkpoint(t, 16)] == [0, 1, 2, 4, 8, 16]
    assert [t for t in range(5) if checkpoint(t, 1)] == [0, 1]
    assert [t for t in range(5) if checkpoint(t, 0)] == [0]


@pytest.mark.parametrize("side", range(3, 11))
def test_finder_matches_brute_force_around_the_settle_time(side):
    """Budgets M at mu + lambda - 1, mu + lambda, mu + lambda + 1, far below and above it, 1 and 0."""
    rs = np.random.RandomState(1000 + side)
    n = 0
    for _ in range(150):
        w = (rs.random_sample(side * side) < rs.choice([0.15, 0.3, 0.5])).astype(np.uint8)
        T = _settle_time(w, side)
        assert T is not None
        budgets = {0, 1, 2, 3, T - 1, T, T + 1, T // 2, 2 * T, T + rs.randint(0, 50), max(0, T - rs.randint(0, 50))}
        for M in sorted(b for b in budgets if b >= 0):
            assert find_settle(w, side, M) == brute_force(w.copy(), side, M), (side, M, T)
            n += 1
    assert n >= 5 * 150                              # about six distinct budgets per board


@pytest.mark.parametrize("rule", [oracle.DEAD_ZERO, oracle.DEAD_DECAY, oracle.DEAD_SAT])
def test_run_settle_leaves_what_brute_force_leaves(rule):
    rs = np.random.RandomState(rule)
    for seed in range(40):
        side = 3 + seed % 8
        w = (rs.random_sample(side * side) < 0.35).astype(np.uint8)
        s = oracle.initial_stable(w, -2)
        args = (-2, 3, rule, -1, -5)
        for M in (0, 1, 7, 60, 400):
            w1, s1, w2, s2 = w.copy(), s.copy(), w.copy(), s.copy()
            got = run_settle(w1, s1, side, -2, 3, M, rule, -1, -5)
            assert got == brute_force(w2, side, M, s2, args), (seed, M)
            assert np.array_equal(w1, w2) and np.array_equal(s1, s2), (seed, M)


@pytest.mark.parametrize("side,cells,period", [(6, GLIDER, 24), (10, GLIDER, 40), (10, LWSS, 20), (12, LWSS, 24), (9, LWSS, 36)])
def test_spaceships_report_their_crossing_period(side, cells, period):
    w = place(side, cells)
    assert find_settle(w, side, 10 * period) == (period, period)
    assert find_settle(w, side, period) == (period, period)        # a match at t == max_steps counts
    assert find_settle(w, side, period - 1) == (period - 1, 0)


def test_a_huge_budget_needs_no_more_than_the_settle_time():
    """The checkpoints below M are powers of two, so a board that settles early is found early at any M."""
    side = 8
    assert find_settle(place(side, [(0, 0), (0, 1), (1, 0), (1, 1)]), side, 2 ** 32 - 1) == (1, 1)
    assert find_settle(place(side, GLIDER), side, 2 ** 32 - 1) == (32, 32)
    assert find_settle(np.zeros(side * side, np.uint8), side, 2 ** 32 - 1) == (1, 1)


def test_env_run_settle_rejects_bad_arguments_without_a_gpu():
    from cgl_b200 import native
    lib = native.load()
    B, k = 4, 8
    plane, world_in, world_out = 0x1000_0000, 0x2000_0000, 0x2100_0000
    acts, rtr, atr, per = 0x3000_0000, 0x3100_0000, 0x3200_0000, 0x3300_0000

    def args(**kw):
        a = native.EnvRunArgs()
        a.world_in, a.world_out, a.stable, a.n_envs, a.side, a.max_steps = world_in, world_out, plane, B, 128, k
        a.spawn, a.stable_max = -1, 1
        a.reward_trace, a.alive_trace = rtr, atr
        for name, v in kw.items():
            setattr(a, name, v)
        return a

    assert lib.cgl_env_run_settle(None, per, None) == native.E_BADARG
    assert b"null" in lib.cgl_last_error()
    cases = [
        (dict(stop_when_fixed=1), b"stop_when_fixed"),
        (dict(actions=acts), b"action schedule"),
        (dict(actions=acts, reward_trace=None, alive_trace=None), b"action schedule"),
        # everything cgl_env_run_ex refuses
        (dict(stable=None), b"bad argument"),
        (dict(world_in=None), b"bad argument"),
        (dict(world_out=None), b"bad argument"),
        (dict(n_envs=0), b"bad argument"),
        (dict(side=0), b"bad argument"),
        (dict(n_envs=1 << 31), b"n_envs too large"),
        (dict(dead_rule=3), b"dead_rule"),
        (dict(dead_rule=-1), b"dead_rule"),
        (dict(empty=128), b"empty"),
        (dict(empty_min=-129), b"empty"),
        (dict(masked_toggle=2), b"masked_toggle"),
        (dict(side=275), b"side <= 274"),
        (dict(side=300), b"side <= 274"),
        (dict(reward_trace=atr), b"separate"),
        (dict(stop_when_fixed=1, actions=acts), b"stop_when_fixed"),
    ]
    for kw, msg in cases:
        a = args(**kw)
        assert lib.cgl_env_run_settle(ctypes.byref(a), per, None) == native.E_BADARG, kw
        assert msg in lib.cgl_last_error(), (kw, lib.cgl_last_error())
    # the shared-memory bound of the other sides, exactly: phase C's three byte planes, 3*side^2 <= 220 KiB (the
    # finder's four bit-vector worlds always fit); it flips between 274 and 275
    fits = [s for s in range(1, 400) if not lib.cgl_env_step_is_fused(s) and 3 * s * s <= 220 * 1024]
    assert max(fits) == 274 and all(4 * 4 * ((s * s + 31) // 32) <= 48 * 1024 for s in fits)
    for side in (275, 276, 299, 301):
        a = args(side=side, reward_trace=None, alive_trace=None)
        assert lib.cgl_env_run_settle(ctypes.byref(a), None, None) == native.E_BADARG, side
        assert b"side <= 274" in lib.cgl_last_error()
