"""Host restatement of cgl_env_run_settle (include/cgl_b200.h, DESIGN.md section 8 f3.4) on the oracle's world step.

world_0 is the world when the call starts and world_t the world after step t.  The run stops after the first step t
(1 <= t <= max_steps) with world_t == world_{t-p} for some 1 <= p <= t and returns (t, p), with no such step
(max_steps, 0).  find_settle restates the device's two world-only phases with their checkpoint schedule and 2M bound;
the tests check it against a brute force that keeps every past world."""
import numpy as np

from oracle import oracle


def checkpoint(t: int, max_steps: int) -> bool:
    """t is in {0} u {2^k < max_steps} u {max_steps}."""
    return t == max_steps or (t < max_steps and t & (t - 1) == 0)


def _life(world: np.ndarray, side: int) -> None:
    """One world-only generation in place (the stability plane does not steer the world)."""
    oracle.step_rule(world, np.zeros(world.size, np.int8), side, -1, 1, oracle.DEAD_ZERO)


def find_settle(world: np.ndarray, side: int, max_steps: int):
    """(steps, period) of one env (uint8 world [side*side], not modified), by phases A and B of the device."""
    M = max_steps
    # A: compare world_t with the checkpoint world_c, c the largest checkpoint below t; give up at t = 2M
    x, ck, c, lam = world.copy(), world, 0, 0
    for i in range(2 * M):
        if checkpoint(i, M):
            ck, c = x.copy(), i
        _life(x, side)
        if np.array_equal(x, ck):
            lam = i + 1 - c
            break
    if lam == 0 or lam > M:
        return M, 0
    # B: runners from world_0 and world_lambda in lockstep; the first equal pair is world_mu
    x, y = world.copy(), world.copy()
    for _ in range(lam):
        _life(y, side)
    mu = 0
    while not np.array_equal(x, y):
        if mu + lam >= M:
            return M, 0
        _life(x, side)
        _life(y, side)
        mu += 1
    return mu + lam, lam


def run_settle(world: np.ndarray, stable: np.ndarray, side: int, spawn: int, stable_max: int, max_steps: int,
               dead_rule: int = 0, empty: int = 0, empty_min: int = -128, on_step=None):
    """Steps ONE env (uint8 world, int8 stable, both [side*side]) in place for the settle run's step count.
    on_step(t, world, stable), if given, is called after every executed step t = 1 .. steps.  Returns (steps, period)."""
    t, p = find_settle(world, side, max_steps)
    for i in range(1, t + 1):
        oracle.step_rule(world, stable, side, spawn, stable_max, dead_rule, empty, empty_min)
        if on_step is not None:
            on_step(i, world, stable)
    return t, p
