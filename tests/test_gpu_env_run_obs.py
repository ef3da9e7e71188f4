"""BatchedSim.run(k, obs_trace=) and TrajectoryReplay.run (cgl_env_run_obs) on the GPU.

Every obs trace is checked plane by plane against k calls of step(actions[t], obs_out=...) from the same start and
against the CPU oracle stepped one action at a time; the rewards, live counts, final world and steps as well.  The
byte kernel serves the fused sides at every k, the generic kernel every other side; CGL_RUN_IMPL does not apply."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import oracle

pytestmark = pytest.mark.gpu

RULES = {"zero": oracle.DEAD_ZERO, "decay": oracle.DEAD_DECAY, "sat": oracle.DEAD_SAT}
FUSED = [32, 64, 96, 128, 160, 192, 224, 256]
OTHER = [1, 10, 17, 100, 200, 274]
RULE_CYCLE = [("zero", False), ("decay", True), ("sat", False), ("zero", True), ("decay", False), ("sat", True)]
# (action schedule, reward and alive traces)
VARIANTS = [(True, True), (True, False), (False, True), (False, False)]


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200 import native
    native.load()
    return torch.device("cuda", 0)


def _env(B, side, rule, masked, spawn, smax, empty, empty_min, seed, **kw):
    from cgl_b200.batched import BatchedSim
    if rule != "zero" or masked:
        kw.update(dead_rule=rule, empty=empty, empty_min=empty_min, masked_toggle=masked)
    return BatchedSim(B, side, seed=seed, spawnStabilityFactor=spawn, stableStabilityFactor=smax, device="cuda:0", **kw)


def _schedule(rs, B, side, k, invalid_env=None):
    size = side * side
    acts = rs.randint(size, size=(k, B)).astype(np.int32)
    acts[rs.rand(k, B) < 0.2] = size                        # no-ops
    if k > 2:
        acts[2] = acts[1]                                   # the same cells twice in a row
    if invalid_env is not None:                             # every other step of one env: out of range
        bad = np.array([-1, size + 1, 1 << 30, -(1 << 31)], np.int32)
        acts[::2, invalid_env] = bad[np.arange(len(acts[::2])) % 4]
    return acts


def oracle_planes(cells, st, side, acts, spawn, smax, rule, empty, empty_min, masked):
    """One env stepped one action at a time: its stability plane after every step; cells / st updated in place."""
    size = side * side
    out = []
    for a in acts:
        a = int(a)
        if 0 <= a < size:
            (oracle.toggle_masked if masked else oracle.toggle)(cells, st, a, spawn)
        oracle.step_rule(cells, st, side, spawn, smax, rule, empty, empty_min)
        out.append(st.copy())
    return np.stack(out) if out else np.zeros((0, size), np.int8)


def _check_case(B, side, k, rule, masked, sched=True, traces=True, factors=(-2, 2, -1, -5), seed=0,
                invalid_env=None):
    spawn, smax, empty, emin = factors
    size = side * side
    rs = np.random.RandomState(seed + side * 7 + k)
    run_env = _env(B, side, rule, masked, spawn, smax, empty, emin, seed)
    step_env = _env(B, side, rule, masked, spawn, smax, empty, emin, seed)
    cells = run_env.get_state().cpu().numpy().copy()
    st = run_env.stable.cpu().numpy().copy()
    src = run_env.stable
    acts = _schedule(rs, B, side, k, invalid_env) if sched else np.full((k, B), size, np.int32)
    acts_d = torch.from_numpy(acts).cuda()
    obs_trace = torch.full((k, B, size), 77, dtype=torch.int8, device="cuda")
    rtrace = torch.full((k, B), -12345, dtype=torch.int32, device="cuda") if traces else None
    atrace = torch.full((k, B), -12345, dtype=torch.int32, device="cuda") if traces else None
    obs, rew, steps = run_env.run(k, want_alive=True, actions=acts_d if sched else None, reward_trace=rtrace,
                                  alive_trace=atrace, obs_trace=obs_trace)
    torch.cuda.synchronize()
    what = f"B={B} side={side} k={k} rule={rule} masked={masked} sched={sched} traces={traces} factors={factors}"
    assert steps.tolist() == [k] * B and run_env.count == k, what
    # out of place: the source plane is untouched and the env's plane is the last row
    assert np.array_equal(src.cpu().numpy(), st), what
    assert obs.data_ptr() == obs_trace[k - 1].data_ptr() and run_env.stable.data_ptr() == obs.data_ptr(), what
    # k single steps with the same actions, each writing its observation to a slot of its own
    ref = torch.full((k, B, size), -77, dtype=torch.int8, device="cuda")
    srew, salv = np.zeros((k, B), np.int64), np.zeros((k, B), np.int64)
    for t in range(k):
        _, r, _ = step_env.step(acts_d[t].contiguous() if sched else None, want_alive=True, obs_out=ref[t])
        srew[t] = r.cpu().numpy()
        salv[t] = step_env.last_alive().cpu().numpy()
    for t in range(k):
        assert torch.equal(obs_trace[t], ref[t]), (what, t)
    if traces:
        assert np.array_equal(rtrace.cpu().numpy(), srew), what
        assert np.array_equal(atrace.cpu().numpy().view(np.uint32), salv), what
    assert torch.equal(run_env.world, step_env.world), what
    assert rew.tolist() == srew[-1].tolist() and run_env.last_alive().tolist() == salv[-1].tolist(), what
    # the oracle, env by env
    got = obs_trace.cpu().numpy()
    for e in range(B):
        planes = oracle_planes(cells[e], st[e], side, acts[:, e], spawn, smax, RULES[rule], empty, emin, masked)
        assert np.array_equal(got[:, e], planes), (what, e)
    assert np.array_equal(run_env.get_state().cpu().numpy(), cells), what
    return run_env, step_env


@pytest.mark.parametrize("k", [1, 2, 3, 4, 63, 257])
@pytest.mark.parametrize("side", FUSED + OTHER)
def test_obs_trace_equals_step_loop_and_oracle(cuda, side, k):
    if k == 257 and side not in (32, 128, 256, 17, 274):
        pytest.skip("257 steps on a subset of sides")
    B = 6 if side <= 64 else 3                             # side <= 64 packs 4 envs per CTA: 6 leaves a partial CTA
    i = (FUSED + OTHER).index(side)
    rule, masked = RULE_CYCLE[i % len(RULE_CYCLE)]
    sched, traces = VARIANTS[(i + [1, 2, 3, 4, 63, 257].index(k)) % len(VARIANTS)]
    _check_case(B, side, k, rule, masked, sched, traces)


@pytest.mark.parametrize("side", [32, 128, 17])
@pytest.mark.parametrize("k", [3, 63])
@pytest.mark.parametrize("rule", ["zero", "decay", "sat"])
@pytest.mark.parametrize("masked", [False, True])
def test_every_dead_rule_with_and_without_masked_toggle(cuda, side, k, rule, masked):
    _check_case(5, side, k, rule, masked, seed=3)


@pytest.mark.parametrize("sched,traces", VARIANTS)
@pytest.mark.parametrize("side", [64, 100])
def test_with_and_without_schedule_and_traces(cuda, side, sched, traces):
    _check_case(5, side, 9, "zero", False, sched, traces, factors=(5, 127, 0, -128), seed=6)


@pytest.mark.parametrize("side,k", [(64, 63), (128, 4), (224, 2), (17, 8)])
def test_invalid_actions_are_ignored_reported_and_traced(cuda, side, k):
    run_env, step_env = _check_case(5, side, k, "zero", False, seed=9, invalid_env=2)
    with pytest.raises(ValueError):
        run_env.check_actions()
    run_env.check_actions()                                # reported once, then cleared
    with pytest.raises(ValueError):
        step_env.check_actions()


@pytest.mark.parametrize("side", [32, 128, 10])
def test_out_of_place_and_zero_steps(cuda, side):
    B = 5
    env = _env(B, side, "zero", False, -2, 2, 0, -128, 1)
    plane = env.stable
    before = plane.clone()
    world = env.world.clone()
    empty = torch.full((0, B, side * side), 9, dtype=torch.int8, device="cuda")
    obs, rew, steps = env.run(0, obs_trace=empty)
    torch.cuda.synchronize()
    assert env.stable.data_ptr() == plane.data_ptr() and torch.equal(plane, before)
    assert torch.equal(env.world, world) and steps.tolist() == [0] * B
    # a k = 0 call with a non-empty buffer writes nothing into it
    from cgl_b200 import native
    buf = torch.full((2, B, side * side), 9, dtype=torch.int8, device="cuda")
    ext = native.ext()
    ext.env_run_ex(env.world, env.stable, side, 0, obs_trace=buf[:0])
    torch.cuda.synchronize()
    assert bool((buf == 9).all()) and torch.equal(plane, before)
    trace = torch.empty((4, B, side * side), dtype=torch.int8, device="cuda")
    obs, _, _ = env.run(4, obs_trace=trace)
    torch.cuda.synchronize()
    assert torch.equal(plane, before), "the source plane was written"
    assert obs.data_ptr() == trace[3].data_ptr() and env.stable.data_ptr() == trace[3].data_ptr()
    # later runs continue from the trace's last row, in place
    env.run(2)
    twin = _env(B, side, "zero", False, -2, 2, 0, -128, 1)
    twin.run(6)
    torch.cuda.synchronize()
    assert env.stable.data_ptr() == trace[3].data_ptr() and torch.equal(trace[3], twin.stable)
    assert torch.equal(env.world, twin.world) and torch.equal(plane, before)


def test_trace_over_4_gib(cuda):
    """4096 x 128^2 for 65 steps: 4.4 GB of trace, rows 64 * 4096 * 16384 bytes = 4 GiB and beyond at the end."""
    from cgl_b200.batched import BatchedSim
    B, side, k = 4096, 128, 65
    size = side * side
    a = BatchedSim(B, side, seed=11, rng="device", device="cuda:0")
    b = BatchedSim(B, side, seed=11, rng="device", device="cuda:0")
    cells0 = a.get_state()
    st0 = a.stable.clone()
    acts = torch.from_numpy(_schedule(np.random.RandomState(5), B, side, k)).cuda()
    trace = torch.empty((k, B, size), dtype=torch.int8, device="cuda")
    assert trace.numel() > (1 << 32)
    a.run(k, actions=acts, obs_trace=trace)
    for t in (k - 2, k - 1):                                # untraced runs from the same start
        b.set_state(cells0)
        b.stable.copy_(st0)
        b.run(t + 1, actions=acts[:t + 1].contiguous())
        assert torch.equal(trace[t], b.stable), t
    assert torch.equal(a.world, b.world)
    envs = [0, 1, 2047, 4095]                               # and single steps for a few envs
    c = BatchedSim(len(envs), side, states=cells0[envs].cpu().numpy(), device="cuda:0")
    c.stable.copy_(st0[envs])
    for t in range(k):
        obs, _, _ = c.step(acts[t, envs].contiguous())
        if t >= k - 3:
            assert torch.equal(trace[t, envs], obs), t
    del trace


_HASH_SCRIPT = r"""
import hashlib, sys
import numpy as np, torch
sys.path[:0] = sys.argv[1:3]
from cgl_b200.batched import BatchedSim
out = []
for side, k in ((32, 2), (128, 3), (128, 9), (256, 5), (17, 6)):
    env = BatchedSim(5, side, seed=side + k, spawnStabilityFactor=-2, stableStabilityFactor=2, device="cuda:0")
    acts = np.random.RandomState(k).randint(side * side + 1, size=(k, 5)).astype(np.int32)
    trace = torch.empty((k, 5, side * side), dtype=torch.int8, device="cuda")
    env.run(k, actions=torch.from_numpy(acts).cuda(), obs_trace=trace)
    out.append(hashlib.sha256(trace.cpu().numpy().tobytes() + env.world.cpu().numpy().tobytes()).hexdigest())
print(" ".join(out))
"""


def test_obs_runs_ignore_the_forced_run_kernel(cuda):
    """CGL_RUN_IMPL picks between the sliced and byte kernels of untraced runs; obs runs give the same bytes."""
    from conftest import PKG, ROOT
    res = {}
    for impl in ("", "bytes", "sliced"):
        env = dict(os.environ, CGL_RUN_IMPL=impl)
        r = subprocess.run([sys.executable, "-c", _HASH_SCRIPT, ROOT, PKG], capture_output=True, text=True, env=env,
                           timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        res[impl] = r.stdout.split()
    assert len(res[""]) == 5 and res[""] == res["bytes"] == res["sliced"]


def test_replay_ring_run_equals_step_loop_across_the_wrap(cuda):
    from cgl_b200.dqn import TrajectoryReplay
    B, side = 6, 64
    mems = []
    for _ in range(2):
        env = _env(B, side, "zero", False, -2, 2, 0, -128, 2)
        mem = TrajectoryReplay(env, max_size=5 * B, batch_size=8, seed=1)
        mem.obs[1:].zero_()
        mems.append(mem)
    ref, got = mems
    assert ref.slots == 6
    rs = np.random.RandomState(4)
    plan = [("step", 2), ("run", 5), ("reset",), ("run", 4), ("run", 1), ("step", 3), ("run", 5), ("run", 3)]
    wrapped = False
    for i, p in enumerate(plan):
        if p[0] == "reset":
            ref.reset()
            got.reset()
        else:
            acts = torch.from_numpy(_schedule(rs, B, side, p[1])).cuda()
            wrapped |= p[0] == "run" and (got.t + 1) % got.slots + p[1] > got.slots
            for t in range(p[1]):
                ref.step(acts[t].contiguous())
            if p[0] == "step":
                for t in range(p[1]):
                    got.step(acts[t].contiguous())
            else:
                got.run(acts)
        torch.cuda.synchronize()
        what = f"after {i}: {p}"
        assert torch.equal(ref.obs, got.obs) and torch.equal(ref.action, got.action), what
        assert torch.equal(ref.reward, got.reward), what
        assert ref.t == got.t and ref._holes == got._holes and ref.size == got.size, what
        assert torch.equal(ref.state, got.state) and got.env.stable.data_ptr() == got.state.data_ptr(), what
        assert torch.equal(ref.env.world, got.env.world), what
    assert wrapped


def test_run_argument_errors(cuda):
    env = _env(4, 32, "zero", False, -1, 1, 0, -128, 0)
    ok = torch.zeros((3, 4, 1024), dtype=torch.int8, device="cuda")
    for bad in (ok.to(torch.int32), ok.cpu(), ok[:, :2], ok.transpose(1, 2).contiguous(), ok.view(3, 4096),
                torch.zeros((6, 4, 1024), dtype=torch.int8, device="cuda")[::2], ok[:2]):
        with pytest.raises(TypeError):
            env.run(3, obs_trace=bad)
    with pytest.raises(ValueError):
        env.run(3, until_fixed=True, obs_trace=ok)
    assert env.count == 0


def test_torch_extension_obs_trace(cuda):
    from cgl_b200 import native
    ext = native.ext()
    for side, k, rule, masked in ((128, 64, "decay", True), (64, 3, "sat", False), (17, 5, "zero", True)):
        B, size = 5, side * side
        a = _env(B, side, rule, masked, -2, 2, -1, -5, 4)
        b = _env(B, side, rule, masked, -2, 2, -1, -5, 4)
        acts = torch.from_numpy(_schedule(np.random.RandomState(k), B, side, k, invalid_env=1)).cuda()
        o1 = torch.zeros((k, B, size), dtype=torch.int8, device="cuda")
        r1, r2 = (torch.zeros((k, B), dtype=torch.int32, device="cuda") for _ in range(2))
        _, rew, steps = a.run(k, actions=acts, reward_trace=r1, obs_trace=o1)
        # the plane and the trace in one buffer, back to back: adjacent is not overlapping
        buf = torch.zeros((k + 1, B, size), dtype=torch.int8, device="cuda")
        buf[0].copy_(b.stable)
        err = torch.zeros(1, dtype=torch.int32, device="cuda")
        rew2 = torch.zeros(B, dtype=torch.int32, device="cuda")
        steps2 = ext.env_run_ex(b.world, buf[0], side, k, False, -2, 2, {"zero": 0, "decay": 1, "sat": 2}[rule], -1,
                                -5, masked, actions=acts, reward_trace=r2, reward_out=rew2, err_flag=err,
                                obs_trace=buf[1:])
        torch.cuda.synchronize()
        assert torch.equal(steps, steps2) and torch.equal(rew, rew2) and torch.equal(r1, r2)
        assert torch.equal(o1, buf[1:]) and torch.equal(buf[0], b.stable)
        assert torch.equal(a.world, b.world)
        assert int(err.item()) == 1
        with pytest.raises(ValueError):
            a.check_actions()
        for bad in (buf[1:].to(torch.int32), buf[1:].cpu(), buf[1:, :2].contiguous(), buf[:k - 1]):
            with pytest.raises(RuntimeError):
                ext.env_run_ex(b.world, buf[0], side, k, False, obs_trace=bad)
        with pytest.raises(RuntimeError):                   # overlaps the plane
            ext.env_run_ex(b.world, buf[1], side, k, False, obs_trace=buf[1:])
        with pytest.raises(RuntimeError, match="stop_when_fixed"):
            ext.env_run_ex(b.world, buf[0], side, k, True, obs_trace=buf[1:])
