"""CPU suite: pin tests/oracle_facade.py, the reference env of tests/test_gpu_single_env_paths.py.

  * OracleEnv replays every golden trace of the reference (base env) and of the fork's CPU back end (dead-cell rule
    "sat", masked toggle, `empty` start) through its facade methods;
  * its seeded start is the reference's; save / load / reset / update_state keep the facade's bookkeeping;
  * the parameter corners cover what the GPU tests rely on.
"""
import numpy as np
import pytest

from conftest import FORK_TRACES, TRACES
from oracle import oracle
from oracle_facade import BASE_CORNERS, CORNERS, EMPTY_PAIRS, OracleEnv, corner_plane


@pytest.mark.parametrize("name", sorted(TRACES))
def test_oracle_env_replays_reference_trace(name):
    tr = TRACES[name]
    env = OracleEnv(tr.worlds[0], tr.stables[0], tr.side, tr.spawn, tr.stable_max)
    assert env.reward() == tr.rewards[0] and env.alive() == tr.alives[0]
    for t in range(tr.T):
        a = tr.action(t)
        if a is not None:
            env.toggle_state(a)
        assert env.reward() == tr.rewards_after_toggle[t], (name, t)
        env.step()
        assert np.array_equal(env.world, tr.worlds[t + 1]) and np.array_equal(env.stable, tr.stables[t + 1]), (name, t)
        assert env.reward() == tr.rewards[t + 1] and env.alive() == tr.alives[t + 1], (name, t)
    assert env.count == tr.T


@pytest.mark.parametrize("name", sorted(FORK_TRACES))
def test_oracle_env_replays_fork_trace(name):
    tr = FORK_TRACES[name]
    world = tr.worlds[0]
    env = OracleEnv(world, oracle.initial_stable_fork(world, tr.spawn, tr.empty), tr.side, tr.spawn, tr.stable_max,
                    oracle.DEAD_SAT, tr.empty, tr.empty_min, masked=True, fork=True)
    assert np.array_equal(env.stable, tr.stables[0])
    for t in range(tr.T):
        a = tr.action(t)
        if a is not None:
            env.toggle_state(a)
        assert np.array_equal(env.stable, tr.toggled_stables[t]), (name, t)
        env.step()
        assert np.array_equal(env.world, tr.worlds[t + 1]) and np.array_equal(env.stable, tr.stables[t + 1]), (name, t)
        assert env.reward() == tr.stability[t + 1] and env.alive() == tr.alives[t + 1], (name, t)


def test_oracle_env_seeded_start_is_the_references():
    tr = TRACES["rand64_plain"]
    env = OracleEnv.seeded(64, 0, -2, 2)
    assert np.array_equal(env.world, tr.worlds[0]) and np.array_equal(env.stable, tr.stables[0])
    fork = OracleEnv.seeded(64, 0, -2, 2, oracle.DEAD_DECAY, -1, -6, masked=True, fork=True)
    assert np.array_equal(fork.stable, np.where(tr.worlds[0] != 0, -2, -1).astype(np.int8))


def test_oracle_env_bookkeeping():
    """reset returns to the start of the current side; a load that keeps the side keeps that start, one that changes
    it starts over from the loaded world; save carries `empty` in the fork only."""
    rs = np.random.RandomState(0)
    env = OracleEnv.seeded(12, 3, -2, 2, oracle.DEAD_SAT, -1, -6, masked=True, fork=True)
    w0, s0 = env.world.copy(), env.stable.copy()
    for _ in range(3):
        env.toggle_state(int(rs.randint(144)))
        env.step()
    sv = env.save()
    assert len(sv) == 7 and sv[3] == 3 and sv[6] == -1
    cells = rs.randint(2, size=144).astype(np.uint8)
    env.load(cells, corner_plane(rs, 144, CORNERS[7]), 12, 40, 5, -1, 3)
    assert (env.count, env.spawn, env.stable_max, env.empty) == (40, 5, -1, 3)
    env.reset()
    assert np.array_equal(env.world, w0) and np.array_equal(env.stable, s0) and env.count == 40
    env.load(cells[:100], np.zeros(100, np.int8), 10, 0, 4, 2, -3)
    env.step()
    env.reset()
    assert np.array_equal(env.world, cells[:100])
    assert np.array_equal(env.stable, np.where(cells[:100] != 0, 4, -3).astype(np.int8))
    base = OracleEnv.seeded(5, 1, -2, 2)
    assert len(base.save()) == 6
    new = rs.randint(2, size=25).astype(np.uint8)
    before = base.stable.copy()
    base.update_state(new)
    assert base.match(new.reshape(5, 5)) and np.array_equal(base.stable, before)


def test_oracle_env_action_rewards_are_brute_force():
    """action_rewards() equals toggle_state(a); step(); reward() for every a, masked and unmasked, on a corner plane."""
    rs = np.random.RandomState(5)
    for corner in (CORNERS[1], CORNERS[9], CORNERS[16]):
        spawn, smax, rule, empty, emin, masked = corner
        world = rs.randint(2, size=36).astype(np.uint8)
        stable = corner_plane(rs, 36, corner)
        env = OracleEnv(world, stable, 6, spawn, smax, rule, empty, emin, masked)
        got = env.action_rewards()
        for a in range(37):
            twin = OracleEnv(world, stable, 6, spawn, smax, rule, empty, emin, masked)
            twin.toggle_state(a)
            twin.step()
            assert got[a] == twin.reward(), (corner, a)


def test_corners_cover_what_the_gpu_tests_need():
    assert len(CORNERS) % 2 and len(CORNERS) % 4            # coprime to 4: side % len meets every side % 4 class
    assert len(set(CORNERS)) == len(CORNERS)
    assert {(c[0], c[1]) for c in BASE_CORNERS} >= {(-2, 2), (-1, -1), (-128, 127), (127, -128), (0, 0), (5, 2)}
    for rule in (oracle.DEAD_DECAY, oracle.DEAD_SAT):
        for e, emin in EMPTY_PAIRS:
            assert {c[5] for c in CORNERS if c[2:5] == (rule, e, emin)} == {False, True}
    # a negative stable_max under every rule, masked and not: what a kernel that drops the sign of max gets wrong
    for rule in (oracle.DEAD_ZERO, oracle.DEAD_DECAY, oracle.DEAD_SAT):
        assert any(c[1] < 0 and c[2] == rule for c in CORNERS)
    assert any(c[1] < 0 and c[5] and c[0] != 0 for c in CORNERS)
    for c in CORNERS:
        assert all(-128 <= v <= 127 for v in c[:5])
