"""CPU suite: the one-step lookahead map (cgl_env_action_rewards).

  * the host restatement (tests/oracle_lookahead.py: the 9-cell formula with every term formed from the step rule,
    by definition on sides 1 and 2) equals brute force -- toggle, step, reward with the oracle -- for every action, on
    sides 1 to 12, all three dead-cell rules, masked and unmasked toggles and constants that wrap int8;
  * the closed forms the kernels run (cgl_bits.cuh lookahead1_rule, built by g++) equal their definition through the
    scalar stability rule, exhaustively over (state, count, stability);
  * every argument error of cgl_env_action_rewards is reported before any device work."""
import ctypes
import os

import numpy as np
import pytest

from conftest import ROOT
from oracle import oracle
import oracle_lookahead as look

TWIN_SRC = os.path.join(ROOT, "tests", "twin", "lookahead_twin.cpp")
_lib = None


def _twin():
    global _lib
    if _lib is None:
        import subprocess
        import tempfile
        out = os.path.join(tempfile.mkdtemp(prefix="cgl_lookahead_twin_"), "liblookahead_twin.so")
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", out, TWIN_SRC], check=True)
        L = ctypes.CDLL(out)
        L.twin_lookahead_mismatches.argtypes = [ctypes.c_int] * 6
        L.twin_lookahead_mismatches.restype = ctypes.c_uint64
        _lib = L
    return _lib


# (spawn, stable_max, empty, empty_min): defaults, a fork setting, and pairs whose SPAWN..MAX range or EMPTY wraps int8
FACTORS = [(-1, 1, 0, -128), (-2, 2, -1, -5), (-128, 127, 127, -128), (127, -128, -128, 127), (5, 127, 126, 3),
           (0, 0, -127, 0)]


def _board(rs, side, density, random_plane):
    world = (rs.rand(side * side) < density).astype(np.uint8)
    stable = (rs.randint(-128, 128, size=side * side) if random_plane else rs.randint(-3, 4, size=side * side))
    return world, stable.astype(np.int8)


@pytest.mark.parametrize("side", range(1, 13))
@pytest.mark.parametrize("rule", [0, 1, 2])
@pytest.mark.parametrize("masked", [False, True])
def test_restatement_equals_brute_force(side, rule, masked):
    rs = np.random.RandomState(side * 7 + rule * 3 + masked)
    for spawn, smax, empty, emin in FACTORS:
        for density, random_plane in ((0.5, True), (0.3, False), (0.0, True), (1.0, True)):
            world, stable = _board(rs, side, density, random_plane)
            want = look.brute_force(world, stable, side, spawn, smax, rule, empty, emin, masked)
            got = look.action_rewards(world, stable, side, spawn, smax, rule, empty, emin, masked)
            assert np.array_equal(got, want), (side, rule, masked, spawn, smax, empty, emin, density)
            assert got[-1] == want[-1]


def test_restatement_wraps_the_sum_like_int32():
    rs = np.random.RandomState(5)
    for side in (2, 7, 12):
        world, stable = _board(rs, side, 0.5, True)
        base = look.brute_force(world, stable, side, -2, 2, 1, -1, -5, True).astype(np.int64)
        for offset in ((1 << 31) - 3, -(1 << 31) + 2, (1 << 32) - 1):
            got = look.action_rewards(world, stable, side, -2, 2, 1, -1, -5, True, offset=offset)
            want = ((base + offset) % (1 << 32)).astype(np.uint32).view(np.int32)
            assert np.array_equal(got, want), (side, offset)


def test_restatement_on_ties_and_still_boards():
    """A block on an empty board: every far cell gives the same reward, so the argmax is the first of a tie."""
    side = 10
    world = np.zeros(side * side, np.uint8)
    for r, c in ((4, 4), (4, 5), (5, 4), (5, 5)):
        world[r * side + c] = 1
    stable = oracle.initial_stable(world, -1)
    got = look.action_rewards(world, stable, side, -1, 1)
    assert np.array_equal(got, look.brute_force(world, stable, side, -1, 1))
    assert (got == got.max()).sum() > 1


@pytest.mark.parametrize("rule", [0, 1, 2])
@pytest.mark.parametrize("masked", [0, 1])
@pytest.mark.parametrize("spawn,smax,empty,emin", FACTORS + [(-2, 3, -100, -90), (3, -128, 2, 10)])
def test_cell_terms_equal_the_scalar_rule_exhaustively(rule, masked, spawn, smax, empty, emin):
    assert _twin().twin_lookahead_mismatches(rule, spawn, smax, empty, emin, masked) == 0


def test_action_rewards_rejects_bad_arguments_without_a_gpu():
    from cgl_b200 import native
    lib = native.load()
    B, side = 4, 128
    size = side * side
    world, plane = 0x1000_0000, 0x2000_0000
    rew, act, best = 0x3000_0000, 0x4000_0000, 0x4100_0000

    def args(**kw):
        a = native.EnvActionRewardsArgs()
        a.world, a.stable, a.n_envs, a.side, a.spawn, a.stable_max = world, plane, B, side, -1, 1
        a.rewards_out, a.best_action_out, a.best_reward_out = rew, act, best
        for name, v in kw.items():
            setattr(a, name, v)
        return a

    assert lib.cgl_env_action_rewards(None, None) == native.E_BADARG
    assert b"null" in lib.cgl_last_error()
    world_bytes, plane_bytes, map_bytes = B * side * 4 * 4, B * size, B * (size + 1) * 4
    cases = [
        (dict(world=None), b"bad argument"),
        (dict(stable=None), b"bad argument"),
        (dict(side=0), b"bad argument"),
        (dict(rewards_out=None, best_action_out=None, best_reward_out=None), b"no output"),
        (dict(n_envs=0), b"n_envs"),
        (dict(n_envs=1 << 31), b"n_envs"),
        (dict(side=46341), b"46340"),
        (dict(dead_rule=3), b"dead_rule"),
        (dict(dead_rule=-1), b"dead_rule"),
        (dict(empty=128), b"empty"),
        (dict(empty=-129), b"empty"),
        (dict(empty_min=128), b"empty"),
        (dict(empty_min=-129), b"empty"),
        (dict(masked_toggle=2), b"masked_toggle"),
        (dict(masked_toggle=-1), b"masked_toggle"),
        # outputs against the inputs: first and last byte of each overlap
        (dict(rewards_out=world + world_bytes - 1), b"overlaps the world or the stability plane"),
        (dict(rewards_out=world - map_bytes + 1), b"overlaps the world or the stability plane"),
        (dict(best_action_out=plane + plane_bytes - 4), b"overlaps the world or the stability plane"),
        (dict(best_reward_out=plane - 3), b"overlaps the world or the stability plane"),
        # outputs against each other
        (dict(best_action_out=rew + map_bytes - 4), b"two outputs overlap"),
        (dict(best_reward_out=act + 2), b"two outputs overlap"),
        (dict(best_reward_out=act), b"two outputs overlap"),
    ]
    for kw, msg in cases:
        a = args(**kw)
        assert lib.cgl_env_action_rewards(ctypes.byref(a), None) == native.E_BADARG, kw
        assert msg in lib.cgl_last_error(), (kw, lib.cgl_last_error())
    # adjacent but disjoint buffers are not an overlap: the call gets past the checks (and then fails on the device,
    # or on the missing device, with a CUDA error -- never with CGL_E_BADARG)
    from cgl_b200.batched import BatchedSim  # noqa: F401
    import torch
    if not torch.cuda.is_available():
        a = args(rewards_out=world + world_bytes, best_action_out=plane + plane_bytes, best_reward_out=rew + map_bytes)
        rc = lib.cgl_env_action_rewards(ctypes.byref(a), None)
        assert rc != 0 and rc != native.E_BADARG


def test_batched_sim_rejects_bad_buffers_without_a_gpu():
    """Argument checks of BatchedSim.action_rewards / greedy_actions run before any device work (on a stand-in
    object: constructing a BatchedSim needs a device)."""
    import torch
    from cgl_b200.batched import BatchedSim
    sim = BatchedSim.__new__(BatchedSim)
    sim.n_envs, sim.side, sim.size, sim.device = 3, 4, 16, torch.device("cpu")
    for bad in (torch.zeros((3, 17), dtype=torch.int64), torch.zeros((3, 16), dtype=torch.int32),
                torch.zeros((17, 3), dtype=torch.int32).t(), "not a tensor"):
        with pytest.raises(TypeError):
            sim.action_rewards(out=bad)
    with pytest.raises(TypeError):
        sim.greedy_actions(out=torch.zeros(4, dtype=torch.int32))
    with pytest.raises(TypeError):
        sim.greedy_actions(reward_out=torch.zeros(3, dtype=torch.int16))
    t = torch.zeros(3, dtype=torch.int32)
    with pytest.raises(TypeError):
        sim.greedy_actions(out=t, reward_out=t)
