"""CPU suite: env runs that stop when the world enters a short cycle (cgl_env_run_cycle).

The host restatement tests/oracle_cycle.py:run_cycle is checked against a brute force that remembers every past world,
and with max_period 1 against the oracle's run-until-fixed on the recorded convergence cases.  The argument checks of
cgl_env_run_cycle run before any device work."""
import ctypes
import json
import os

import numpy as np
import pytest

from oracle import oracle
from oracle_cycle import run_cycle

HERE = os.path.dirname(os.path.abspath(__file__))
with open(os.path.join(HERE, "golden", "golden_converge.json")) as f:
    CONVERGE = [c for c in json.load(f)["cases"] if c["mode"] == "converge"]

PULSAR = [rc for r in (0, 5, 7, 12) for c in (2, 3, 4, 8, 9, 10) for rc in ((r, c), (c, r))]          # period 3
FIGURE_EIGHT = [(r, c) for r in range(3) for c in range(3)] + [(r + 3, c + 3) for r in range(3) for c in range(3)]


def place(side, cells, r0=2, c0=2):
    w = np.zeros(side * side, dtype=np.uint8)
    for r, c in cells:
        w[((r0 + r) % side) * side + (c0 + c) % side] = 1
    return w


def brute_force(world, stable, side, spawn, stable_max, max_steps, max_period, dead_rule=0, empty=0,
                empty_min=-128):
    """Every past world in a dict; the first step whose world was seen at most max_period steps ago."""
    seen = {world.tobytes(): 0}
    for t in range(1, max_steps + 1):
        oracle.step_rule(world, stable, side, spawn, stable_max, dead_rule, empty, empty_min)
        k = world.tobytes()
        if k in seen and t - seen[k] <= max_period:
            return t, t - seen[k]
        seen[k] = t
    return max_steps, 0


def _boards(seed, side):
    rs = np.random.RandomState(seed)
    w = (rs.random_sample(side * side) < rs.choice([0.2, 0.35, 0.5])).astype(np.uint8)
    return w, oracle.initial_stable(w, -2)


@pytest.mark.parametrize("side", range(1, 13))
def test_run_cycle_matches_brute_force_on_random_tori(side):
    for seed in range(12):
        for P in range(1, 9):
            for rule in (oracle.DEAD_ZERO, oracle.DEAD_DECAY, oracle.DEAD_SAT):
                w0, s0 = _boards(seed, side)
                args = (side, -2, 3, 200, P, rule, -1, -5)
                w1, s1, w2, s2 = w0.copy(), s0.copy(), w0.copy(), s0.copy()
                got = run_cycle(w1, s1, *args)
                ref = brute_force(w2, s2, *args)
                assert got == ref, (side, seed, P, rule)
                assert np.array_equal(w1, w2) and np.array_equal(s1, s2)


def _soup(side, seed, density, index=0, batch=1):
    rs = np.random.RandomState(seed)
    return (rs.random_sample((batch, side * side)) < density).astype(np.uint8)[index]


# One board of each period: (side, world).  Random soups on small tori (found by a search over seeds) where they give
# the period, known oscillators where they do not: the pulsar (3) and the figure eight (8).
PERIODIC_BOARDS = {
    1: (3, _soup(3, 0, 0.5)),
    2: (4, _soup(4, 0, 0.5)),
    3: (20, place(20, PULSAR)),
    4: (4, _soup(4, 219, 0.3)),
    5: (5, _soup(5, 5050, 0.5, index=679, batch=4000)),
    6: (6, _soup(6, 338, 0.3)),
    8: (12, place(12, FIGURE_EIGHT)),
}


def _world_period(w, side, limit=200):
    """The exact period of the cycle the world enters (every past world kept), or None."""
    seen, s, w = {w.tobytes(): 0}, np.zeros(w.size, np.int8), w.copy()
    for t in range(1, limit):
        oracle.step_rule(w, s, side, -1, 1, 0)
        if w.tobytes() in seen:
            return t - seen[w.tobytes()]
        seen[w.tobytes()] = t
    return None


@pytest.mark.parametrize("p", sorted(PERIODIC_BOARDS))
def test_each_period_is_found_exactly(p):
    side, w = PERIODIC_BOARDS[p]
    assert _world_period(w, side) == p
    for P in range(1, 9):
        w1, s1 = w.copy(), oracle.initial_stable(w, -1)
        w2, s2 = w.copy(), s1.copy()
        got = run_cycle(w1, s1, side, -1, 1, 300, P)
        assert got == brute_force(w2, s2, side, -1, 1, 300, P), (p, P)
        assert got[1] == (p if P >= p else 0), (p, P, got)


def test_period_is_unique_and_is_the_cycle_length():
    """The matched lag is the only lag <= P at which world_t repeats, and the world then repeats every p steps."""
    for seed in range(40):
        side = 4 + seed % 9
        w, s = _boards(seed, side)
        for P in (2, 3, 8):
            w1, s1 = w.copy(), s.copy()
            hist = [w1.copy()]
            t, p = run_cycle(w1, s1, side, -2, 3, 500, P, on_step=lambda t, ww, ss: hist.append(ww.copy()))
            assert len(hist) == t + 1
            if p == 0:
                continue
            assert [q for q in range(1, min(P, t) + 1) if np.array_equal(hist[t], hist[t - q])] == [p]
            for i in range(max(0, t - P), t):                  # the window before the stop is pairwise distinct
                for j in range(i + 1, t):
                    assert not np.array_equal(hist[i], hist[j])
            w2 = w1.copy()
            for _ in range(p):
                oracle.step_rule(w2, np.zeros_like(s1), side, -2, 3, 0)
            assert np.array_equal(w2, w1)


def test_match_at_the_last_step_counts():
    side = 12
    w = place(side, FIGURE_EIGHT)
    t, p = run_cycle(w.copy(), oracle.initial_stable(w, -1), side, -1, 1, 8, 8)
    assert (t, p) == (8, 8)
    assert run_cycle(w.copy(), oracle.initial_stable(w, -1), side, -1, 1, 7, 8) == (7, 0)
    assert run_cycle(w.copy(), oracle.initial_stable(w, -1), side, -1, 1, 0, 8) == (0, 0)


@pytest.mark.parametrize("c", CONVERGE, ids=lambda c: f"side{c['side']}-seed{c['seed']}")
def test_period_1_equals_run_until_fixed_on_the_recorded_cases(c):
    w1 = oracle.initial_world(c["side"], c["seed"])
    s1 = oracle.initial_stable(w1, c["spawn"])
    w2, s2 = w1.copy(), s1.copy()
    n = oracle.run(w1, s1, c["side"], c["spawn"], c["stable"], c["limit"] + 1, until_fixed=True)
    t, p = run_cycle(w2, s2, c["side"], c["spawn"], c["stable"], c["limit"] + 1, 1)
    assert t == n == c["steps"] and p in (0, 1)
    if t < c["limit"] + 1:
        assert p == 1
    assert np.array_equal(w1, w2) and np.array_equal(s1, s2)


def test_env_run_cycle_rejects_bad_arguments_without_a_gpu():
    from cgl_b200 import native
    lib = native.load()
    assert native.RUN_MAX_PERIOD == 8
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

    assert lib.cgl_env_run_cycle(None, 2, per, None) == native.E_BADARG
    assert b"null" in lib.cgl_last_error()
    cases = [
        (dict(stop_when_fixed=1), 2, b"stop_when_fixed"),
        (dict(actions=acts), 2, b"action schedule"),
        (dict(), 0, b"max_period"),
        (dict(), 9, b"max_period"),
        (dict(side=269), 1, b"side <= 268 at max_period 1"),
        (dict(side=238), 8, b"<= 237 at 8"),
        (dict(side=237), 9, b"max_period"),
        # everything cgl_env_run_ex refuses
        (dict(stable=None), 2, b"bad argument"),
        (dict(world_in=None), 2, b"bad argument"),
        (dict(n_envs=0), 2, b"bad argument"),
        (dict(side=0), 2, b"bad argument"),
        (dict(n_envs=1 << 31), 2, b"n_envs too large"),
        (dict(dead_rule=3), 2, b"dead_rule"),
        (dict(dead_rule=-1), 2, b"dead_rule"),
        (dict(empty=128), 2, b"empty"),
        (dict(empty_min=-129), 2, b"empty"),
        (dict(masked_toggle=2), 2, b"masked_toggle"),
        (dict(side=275), 2, b"side <= 274"),
        (dict(reward_trace=atr), 2, b"separate"),
        (dict(stop_when_fixed=1, actions=acts), 2, b"stop_when_fixed"),
    ]
    for kw, P, msg in cases:
        a = args(**kw)
        assert lib.cgl_env_run_cycle(ctypes.byref(a), P, per, None) == native.E_BADARG, (kw, P)
        assert msg in lib.cgl_last_error(), (kw, P, lib.cgl_last_error())
    # the bound of the generic kernel, exactly: 3*side^2 (rounded up to 4) + P*4*ceil(side^2/32) <= 220 KiB
    for P in range(1, 9):
        fits = [s for s in range(1, 300) if ((3 * s * s + 3) & ~3) + P * 4 * ((s * s + 31) // 32) <= 220 * 1024]
        assert fits == list(range(1, max(fits) + 1))
        assert max(fits) == {1: 268, 8: 237}.get(P, max(fits))
        a = args(side=max(fits) + 1, reward_trace=None, alive_trace=None)
        if not native.load().cgl_env_step_is_fused(max(fits) + 1):
            assert lib.cgl_env_run_cycle(ctypes.byref(a), P, per, None) == native.E_BADARG, P
            assert b"220 KiB" in lib.cgl_last_error()
