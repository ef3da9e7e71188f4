"""BatchedSim.run with an action schedule and per-step reward / alive traces (cgl_env_run_ex) on the GPU.

Every case is checked three ways: against k calls of step(actions[t]) with the reward and live count read after each,
against the CPU oracle stepped one action at a time, and for the final world, stability plane, reward, alive and steps.
The three run kernels are reached through the side (fused sides 32..256, any other side <= 274) and the step count
(the byte kernel below 4 steps, the bit-sliced one from 4 on); each is also forced for every step count in a fresh
process with CGL_RUN_IMPL."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import oracle
from test_env_run_actions_cpu import oracle_run

pytestmark = pytest.mark.gpu

RULES = {"zero": oracle.DEAD_ZERO, "decay": oracle.DEAD_DECAY, "sat": oracle.DEAD_SAT}


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200 import native
    native.load()
    return torch.device("cuda", 0)


def _env(B, side, rule, masked, spawn, smax, empty, empty_min, seed):
    from cgl_b200.batched import BatchedSim
    kw = {} if rule == "zero" and not masked else dict(dead_rule=rule, empty=empty, empty_min=empty_min,
                                                       masked_toggle=masked)
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


def _check_case(B, side, k, rule, masked, factors=(-2, 2, -1, -5), seed=0, invalid_env=None):
    spawn, smax, empty, emin = factors
    rs = np.random.RandomState(seed + side * 7 + k)
    run_env = _env(B, side, rule, masked, spawn, smax, empty, emin, seed)
    step_env = _env(B, side, rule, masked, spawn, smax, empty, emin, seed)
    cells = run_env.get_state().cpu().numpy().copy()
    st = run_env.stable.cpu().numpy().copy()
    acts = _schedule(rs, B, side, k, invalid_env)
    acts_d = torch.from_numpy(acts).cuda()
    rtrace = torch.full((k, B), -12345, dtype=torch.int32, device="cuda")
    atrace = torch.full((k, B), -12345, dtype=torch.int32, device="cuda")
    obs, rew, steps = run_env.run(k, want_alive=True, actions=acts_d, reward_trace=rtrace, alive_trace=atrace)
    torch.cuda.synchronize()
    what = f"B={B} side={side} k={k} rule={rule} masked={masked} factors={factors}"
    assert steps.tolist() == [k] * B and run_env.count == k, what
    # k single steps with the same actions
    srew, salv = np.zeros((k, B), np.int64), np.zeros((k, B), np.int64)
    for t in range(k):
        _, r, _ = step_env.step(acts_d[t].contiguous(), want_alive=True)
        srew[t] = r.cpu().numpy()
        salv[t] = step_env.last_alive().cpu().numpy()
    assert np.array_equal(rtrace.cpu().numpy(), srew), what
    assert np.array_equal(atrace.cpu().numpy().view(np.uint32), salv), what
    assert torch.equal(run_env.world, step_env.world) and torch.equal(obs, step_env.stable), what
    # the oracle, env by env
    for e in range(B):
        r_o, a_o = oracle_run(cells[e], st[e], side, acts[:, e], spawn, smax, RULES[rule], empty, emin, masked)
        assert rtrace[:, e].tolist() == r_o, (what, e)
        assert atrace[:, e].cpu().numpy().view(np.uint32).tolist() == a_o, (what, e)
    assert np.array_equal(run_env.get_state().cpu().numpy(), cells), what
    assert np.array_equal(obs.cpu().numpy(), st), what
    assert rew.tolist() == rtrace[-1].tolist() and run_env.last_alive().tolist() == atrace[-1].tolist(), what
    return run_env, step_env


FUSED = [32, 64, 96, 128, 160, 192, 224, 256]
GENERIC = [10, 17, 100, 200, 274]
RULE_CYCLE = [("zero", False), ("decay", True), ("sat", False), ("zero", True), ("decay", False), ("sat", True)]


@pytest.mark.parametrize("k", [1, 2, 3, 4, 64, 257])
@pytest.mark.parametrize("side", FUSED + GENERIC)
def test_run_with_actions_equals_step_loop_and_oracle(cuda, side, k):
    if k == 257 and side not in (32, 128, 256, 17, 274):
        pytest.skip("257 steps on a subset of sides")
    B = 6 if side <= 64 else 3                             # side <= 64 packs 4 envs per CTA: 6 leaves a partial CTA
    rule, masked = RULE_CYCLE[(FUSED + GENERIC).index(side) % len(RULE_CYCLE)]
    _check_case(B, side, k, rule, masked)


@pytest.mark.parametrize("side", [32, 128, 17])
@pytest.mark.parametrize("k", [3, 64])
@pytest.mark.parametrize("rule", ["zero", "decay", "sat"])
@pytest.mark.parametrize("masked", [False, True])
def test_every_dead_rule_with_and_without_masked_toggle(cuda, side, k, rule, masked):
    _check_case(5, side, k, rule, masked, seed=3)


@pytest.mark.parametrize("factors", [(5, 127, 0, -128), (100, -100, -3, -20), (-1, 1, 0, -128)])
@pytest.mark.parametrize("side", [64, 128])
def test_spawn_max_pairs_that_wrap_int8(cuda, factors, side):
    for rule in ("zero", "decay", "sat"):
        _check_case(6, side, 40, rule, False, factors=factors, seed=5)


@pytest.mark.parametrize("side,k", [(64, 64), (128, 64), (128, 2), (17, 8)])
def test_invalid_actions_are_ignored_reported_and_leave_other_envs_alone(cuda, side, k):
    run_env, step_env = _check_case(5, side, k, "zero", False, seed=9, invalid_env=2)
    with pytest.raises(ValueError):
        run_env.check_actions()
    run_env.check_actions()                                # reported once, then cleared
    with pytest.raises(ValueError):
        step_env.check_actions()


@pytest.mark.parametrize("side", [32, 128, 17])
@pytest.mark.parametrize("impl_k", [2, 40])
def test_traces_under_until_fixed_stop_at_each_envs_fixed_point(cuda, side, impl_k):
    B, spawn, smax = 6, -1, 1
    env = _env(B, side, "zero", False, spawn, smax, 0, -128, 0)
    # mostly empty worlds settle within a few steps; env 0 keeps its random start
    cells = env.get_state().cpu().numpy().copy()
    cells[1:] *= (np.random.RandomState(1).rand(B - 1, side * side) < 0.08).astype(np.uint8)
    cells[1] = 0                                            # fixed from the start: one step
    env.set_state(torch.from_numpy(cells).cuda())
    env.init_stable()
    st = env.stable.cpu().numpy().copy()
    k = impl_k
    rtrace = torch.full((k, B), -777, dtype=torch.int32, device="cuda")
    atrace = torch.full((k, B), -777, dtype=torch.int32, device="cuda")
    _, rew, steps = env.run(k, until_fixed=True, reward_trace=rtrace, alive_trace=atrace)
    steps = steps.tolist()
    for e in range(B):
        w, s = cells[e].copy(), st[e].copy()
        n = oracle.run(w, s, side, spawn, smax, k, True)
        assert steps[e] == n
        w, s = cells[e].copy(), st[e].copy()
        r_o, a_o = oracle_run(w, s, side, [side * side] * n, spawn, smax, oracle.DEAD_ZERO, 0, -128, False)
        assert rtrace[:n, e].tolist() == r_o and atrace[:n, e].tolist() == a_o, e
        assert rtrace[n:, e].tolist() == [-777] * (k - n) and atrace[n:, e].tolist() == [-777] * (k - n), e
        if n:
            assert int(rew[e]) == r_o[-1]
    assert min(steps) < k                                   # some env did stop early


def test_run_argument_errors(cuda):
    env = _env(4, 32, "zero", False, -1, 1, 0, -128, 0)
    ok = torch.zeros((3, 4), dtype=torch.int32, device="cuda")
    for bad in (ok.to(torch.int64), ok.cpu(), ok.t().contiguous(), ok[:, :2], torch.zeros((6, 4), dtype=torch.int32,
                                                                                          device="cuda")[::2]):
        for name in ("actions", "reward_trace", "alive_trace"):
            with pytest.raises(TypeError):
                env.run(3, **{name: bad})
    with pytest.raises(ValueError):
        env.run(3, until_fixed=True, actions=ok)
    assert env.count == 0


def test_torch_extension_env_run_ex_equals_ctypes_path(cuda):
    from cgl_b200 import native
    ext = native.ext()
    for side, k, rule, masked in ((128, 64, "decay", True), (64, 3, "sat", False), (17, 5, "zero", True)):
        B = 5
        a = _env(B, side, rule, masked, -2, 2, -1, -5, 4)
        b = _env(B, side, rule, masked, -2, 2, -1, -5, 4)
        acts = torch.from_numpy(_schedule(np.random.RandomState(k), B, side, k, invalid_env=1)).cuda()
        r1, a1 = (torch.zeros((k, B), dtype=torch.int32, device="cuda") for _ in range(2))
        r2, a2 = (torch.zeros((k, B), dtype=torch.int32, device="cuda") for _ in range(2))
        _, rew, steps = a.run(k, actions=acts, reward_trace=r1, alive_trace=a1)
        err = torch.zeros(1, dtype=torch.int32, device="cuda")
        rew2 = torch.zeros(B, dtype=torch.int32, device="cuda")
        steps2 = ext.env_run_ex(b.world, b.stable, side, k, False, -2, 2, {"zero": 0, "decay": 1, "sat": 2}[rule], -1,
                                -5, masked, actions=acts, reward_trace=r2, alive_trace=a2, reward_out=rew2,
                                err_flag=err)
        torch.cuda.synchronize()
        assert torch.equal(steps, steps2) and torch.equal(rew, rew2)
        assert torch.equal(r1, r2) and torch.equal(a1, a2)
        assert torch.equal(a.world, b.world) and torch.equal(a.stable, b.stable)
        assert int(err.item()) == 1
        with pytest.raises(ValueError):
            a.check_actions()
        with pytest.raises(RuntimeError):
            ext.env_run_ex(b.world, b.stable, side, k, False, actions=acts[:, :2].contiguous())


@pytest.mark.parametrize("impl", ["bytes", "sliced"])
def test_both_run_kernels_follow_the_schedule(cuda, impl):
    """Each in-SM kernel forced for every step count and side of the main test, in a fresh process."""
    env = dict(os.environ, CGL_RUN_IMPL=impl)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-x", "-k",
                        "test_run_with_actions_equals_step_loop_and_oracle and not 257"],
                       capture_output=True, text=True, env=env, timeout=1500)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
