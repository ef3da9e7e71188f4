"""CPU suite: env runs that record every step's observation (cgl_env_run_obs) and the replay ring filled by them.

The argument checks of cgl_env_run_obs run before any device work.  TrajectoryReplay.run is checked against k calls of
TrajectoryReplay.step on the CPU oracle env, whose run() steps the oracle one action at a time into the obs trace."""
import ctypes

import numpy as np
import pytest

from oracle import oracle

torch = pytest.importorskip("torch")

from cgl_b200.dqn import TrajectoryReplay  # noqa: E402
from oracle_env import OracleBatchEnv  # noqa: E402


class OracleRunEnv(OracleBatchEnv):
    """OracleBatchEnv with BatchedSim.run(k, actions=, reward_trace=, obs_trace=): out of place, one action at a time."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.runs = []

    def run(self, max_steps, actions=None, reward_trace=None, obs_trace=None):
        assert obs_trace.shape == (max_steps, self.n_envs, self.size) and obs_trace.is_contiguous()
        assert actions.shape == (max_steps, self.n_envs) and reward_trace.shape == (max_steps, self.n_envs)
        lo, hi = obs_trace.data_ptr(), obs_trace.data_ptr() + obs_trace.numel()
        assert not lo <= self.stable.data_ptr() < hi, "the obs trace must not hold the live plane"
        src = self.stable.clone()
        for t in range(max_steps):
            obs_trace[t].copy_(src)
            rew, _ = oracle.step_batch(self.world, obs_trace[t].numpy(), self.side, actions[t].numpy(), self.spawn,
                                       self.stable_max)
            reward_trace[t] = torch.from_numpy(rew)
            src = obs_trace[t]
        if max_steps:
            self.stable = obs_trace[max_steps - 1]
        self.runs.append(max_steps)
        return self.stable, None, None


def _pair(B=3, side=6, slots=5, seed=2):
    """Two replays over identical envs; unwritten obs slots zeroed so that whole rings compare."""
    out = []
    for _ in range(2):
        env = OracleRunEnv(B, side, seed=seed)
        mem = TrajectoryReplay(env, max_size=(slots - 1) * B, batch_size=4, seed=1)
        assert mem.slots == slots
        mem.obs[1:].zero_()
        out.append((env, mem))
    return out


def _acts(rs, k, B, side):
    a = rs.randint(0, side * side + 1, size=(k, B)).astype(np.int32)
    return torch.from_numpy(a)


def _assert_same(ref, got, what):
    (env_a, a), (env_b, b) = ref, got
    assert torch.equal(a.obs, b.obs), what
    assert torch.equal(a.action, b.action), what
    assert torch.equal(a.reward, b.reward), what
    assert a.t == b.t and a._holes == b._holes and a.valid_steps() == b.valid_steps() and a.size == b.size, what
    assert torch.equal(a.state, b.state), what
    assert b.env.stable.data_ptr() == b.state.data_ptr() and a.env.stable.data_ptr() == a.state.data_ptr(), what
    assert np.array_equal(env_a.world, env_b.world), what


def _step_loop(mem, acts):
    out = None
    for i in range(acts.shape[0]):
        out = mem.step(acts[i].clone())
    return out


@pytest.mark.parametrize("offset", range(5))
def test_run_equals_step_loop_at_every_ring_offset(offset):
    slots, B, side = 5, 3, 6
    for k in range(1, slots):
        ref, got = _pair(B, side, slots)
        rs = np.random.RandomState(offset * 10 + k)
        pre = _acts(rs, offset, B, side)
        _step_loop(ref[1], pre)
        _step_loop(got[1], pre)
        acts = _acts(rs, k, B, side)
        n_ref, r_ref = _step_loop(ref[1], acts)
        n_got, r_got = got[1].run(acts)
        what = f"offset={offset} k={k}"
        _assert_same(ref, got, what)
        assert n_got.data_ptr() - got[1].obs.data_ptr() == n_ref.data_ptr() - ref[1].obs.data_ptr(), what
        assert r_got.data_ptr() - got[1].reward.data_ptr() == r_ref.data_ptr() - ref[1].reward.data_ptr(), what
        o = (offset + 1) % slots
        assert got[0].runs == ([k] if o + k <= slots else [slots - o, k - (slots - o)]), what


def test_runs_after_reset_leave_the_same_holes():
    ref, got = _pair(B=2, side=5, slots=6, seed=4)
    rs = np.random.RandomState(7)
    plan = [("run", 3), ("reset",), ("run", 5), ("step", 2), ("reset",), ("reset",), ("run", 4), ("run", 1),
            ("reset",), ("run", 5), ("step", 1), ("reset",), ("run", 2), ("step", 1)]
    for i, p in enumerate(plan):
        if p[0] == "reset":
            ref[1].reset()
            got[1].reset()
        else:
            acts = _acts(rs, p[1], 2, 5)
            _step_loop(ref[1], acts)
            (_step_loop if p[0] == "step" else lambda m, a: m.run(a))(got[1], acts)
        _assert_same(ref, got, f"after {i}: {p}")
    assert got[1]._holes and got[1].size == ref[1].size
    for _ in range(3):                                     # sampling sees the same transitions
        sa, sb = ref[1].sample(), got[1].sample()
        for x, y in zip(sa, sb):
            assert torch.equal(x, y)


def test_run_k_bounds():
    (_, mem), _ = _pair(B=3, side=6, slots=5)
    rs = np.random.RandomState(0)
    for k in (0, 5, 9):
        with pytest.raises(ValueError):
            mem.run(torch.zeros((k, 3), dtype=torch.int32))
    assert mem.t == 0
    with pytest.raises(TypeError):
        mem.run(torch.zeros((2, 4), dtype=torch.int32))
    with pytest.raises(TypeError):
        mem.run([[0, 0, 0]])
    ref, got = _pair(B=3, side=6, slots=5)
    _step_loop(ref[1], _acts(np.random.RandomState(1), 2, 3, 6))
    _step_loop(got[1], _acts(np.random.RandomState(1), 2, 3, 6))
    acts = _acts(rs, 4, 3, 6)                              # k = slots - 1: every resident step is new
    _step_loop(ref[1], acts)
    got[1].run(acts)
    _assert_same(ref, got, "k = slots - 1")


def test_env_run_obs_rejects_bad_arguments_without_a_gpu():
    from cgl_b200 import native
    lib = native.load()
    B, side, k = 4, 128, 8
    size = side * side
    plane, world_in, world_out = 0x1000_0000, 0x2000_0000, 0x2100_0000
    acts, rtr, atr, obs = 0x3000_0000, 0x3100_0000, 0x3200_0000, 0x4000_0000
    obs_bytes = k * B * size

    def args(obs_trace=obs, **kw):
        a = native.EnvRunObsArgs()
        r = a.run
        r.world_in, r.world_out, r.stable, r.n_envs, r.side, r.max_steps = world_in, world_out, plane, B, side, k
        r.spawn, r.stable_max = -1, 1
        r.actions, r.reward_trace, r.alive_trace = acts, rtr, atr
        for name, v in kw.items():
            setattr(r, name, v)
        a.obs_trace = obs_trace
        return a

    assert lib.cgl_env_run_obs(None, None) == native.E_BADARG
    assert b"null" in lib.cgl_last_error()
    cases = [
        (dict(stop_when_fixed=1, actions=None), b"stop_when_fixed"),
        (dict(obs_trace=plane), b"overlaps"),                                   # the plane itself
        (dict(obs_trace=plane - obs_bytes + 1), b"overlaps"),                   # its last byte on the plane's first
        (dict(obs_trace=plane + B * size - 16), b"overlaps"),                   # starts inside the plane
        (dict(obs_trace=acts - obs_bytes + 16), b"overlaps"),                   # ends inside the schedule
        (dict(obs_trace=rtr + 4 * k * B - 16), b"overlaps"),                    # starts in the reward trace's tail
        (dict(obs_trace=atr + 64), b"overlaps"),
        (dict(obs_trace=world_out - 16), b"overlaps"),
        (dict(obs_trace=obs + 8), b"16-byte aligned"),                          # fused side
        (dict(stable=None), b"bad argument"),
        (dict(dead_rule=3), b"dead_rule"),
        (dict(masked_toggle=2), b"masked_toggle"),
        (dict(side=275), b"side <= 274"),
        (dict(reward_trace=atr), b"separate"),
        (dict(stop_when_fixed=1), b"stop_when_fixed"),                          # with actions: the older check
    ]
    for kw, msg in cases:
        a = args(**kw)
        assert lib.cgl_env_run_obs(ctypes.byref(a), None) == native.E_BADARG, kw
        assert msg in lib.cgl_last_error(), (kw, lib.cgl_last_error())
    # 64-bit trace sizes: 4096 envs x 128^2 x 65 steps is 4.4 GB; a trace that reaches the plane from below is refused
    big = args(n_envs=4096, max_steps=65, actions=None, reward_trace=None, alive_trace=None,
               stable=0x2_0000_0000, world_in=0x3_0000_0000, world_out=0x3_0000_0000,
               obs_trace=0x2_0000_0000 - 65 * 4096 * size + (1 << 32) - 16)
    assert lib.cgl_env_run_obs(ctypes.byref(big), None) == native.E_BADARG
    assert b"overlaps" in lib.cgl_last_error()
