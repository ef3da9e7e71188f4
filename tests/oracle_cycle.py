"""Host restatement of cgl_env_run_cycle (include/cgl_b200.h) on top of the oracle's single step.

world_0 is the world when the call starts and world_t the world after step t.  The run stops after the first step t
(1 <= t <= max_steps) with world_t == world_{t-p} for some 1 <= p <= min(max_period, t), and returns (t, p); with no
such step it returns (max_steps, 0).  Only the world is compared; the stability plane follows its own rule."""
from collections import deque

import numpy as np

from oracle import oracle


def run_cycle(world: np.ndarray, stable: np.ndarray, side: int, spawn: int, stable_max: int, max_steps: int,
              max_period: int, dead_rule: int = 0, empty: int = 0, empty_min: int = -128, on_step=None):
    """Steps ONE env (uint8 world, int8 stable, both [side*side]) in place.  on_step(t, world, stable), if given,
    is called after every executed step t = 1 .. steps.  Returns (steps, period)."""
    assert 1 <= max_period
    past = deque([world.tobytes()], maxlen=max_period)     # past[-p] = world_{t-p} before step t
    t = 0
    while t < max_steps:
        oracle.step_rule(world, stable, side, spawn, stable_max, dead_rule, empty, empty_min)
        t += 1
        if on_step is not None:
            on_step(t, world, stable)
        cur = world.tobytes()
        for p in range(1, len(past) + 1):
            if past[-p] == cur:
                return t, p
        past.append(cur)
    return t, 0
