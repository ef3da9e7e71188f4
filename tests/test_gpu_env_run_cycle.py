"""BatchedSim.run(k, max_period=) and the facades' run_until_cycle (cgl_env_run_cycle) on the GPU.

  * max_period = 1 equals until_fixed in every output, on every fused side and on generic sides;
  * every recorded convergence case is reproduced through max_period = 1;
  * batches of known oscillators, a glider and random soups agree with tests/oracle_cycle.py:run_cycle env by env,
    trace rows from steps[e] on untouched;
  * the bounds: a match at the last step, the generic kernel's shared-memory bound, CGL_RUN_IMPL, argument errors."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import oracle
from oracle_cycle import run_cycle

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
with open(os.path.join(HERE, "golden", "golden_converge.json")) as f:
    CONVERGE = [c for c in json.load(f)["cases"] if c["mode"] == "converge"]

RULES = {"zero": oracle.DEAD_ZERO, "decay": oracle.DEAD_DECAY, "sat": oracle.DEAD_SAT}
FUSED = [32, 64, 96, 128, 160, 192, 224, 256]
GENERIC = [1, 2, 3, 10, 17, 33, 100, 200]
FACTORS = (-2, 2, -1, -5)                     # spawn, stable_max, empty, empty_min
SENTINEL = -12345

BLOCK = [(0, 0), (0, 1), (1, 0), (1, 1)]
BLINKER = [(0, 0), (0, 1), (0, 2)]
PULSAR = [rc for r in (0, 5, 7, 12) for c in (2, 3, 4, 8, 9, 10) for rc in ((r, c), (c, r))]          # period 3
FIGURE_EIGHT = [(r, c) for r in range(3) for c in range(3)] + [(r + 3, c + 3) for r in range(3) for c in range(3)]
GLIDER = [(0, 1), (1, 2), (2, 0), (2, 1), (2, 2)]


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200 import native
    native.load()
    return torch.device("cuda", 0)


def place(side, cells, r0=2, c0=2):
    w = np.zeros(side * side, dtype=np.uint8)
    for r, c in cells:
        w[((r0 + r) % side) * side + (c0 + c) % side] = 1
    return w


def _env(cells, side, rule):
    from cgl_b200.batched import BatchedSim
    spawn, smax, empty, emin = FACTORS
    kw = {} if rule == "zero" else dict(dead_rule=rule, empty=empty, empty_min=emin)
    env = BatchedSim(len(cells), side, spawnStabilityFactor=spawn, stableStabilityFactor=smax, device="cuda:0",
                     rng="device", **kw)
    env.set_state(torch.from_numpy(np.ascontiguousarray(cells)).cuda())
    env.init_stable()
    return env


def _soups(rs, n, side):
    dens = rs.choice([0.05, 0.15, 0.3, 0.5], size=n)
    return (rs.random_sample((n, side * side)) < dens[:, None]).astype(np.uint8)


def _run(env, k, **kw):
    """run(k, ...) with sentinel-filled traces; returns (steps, world, stable, reward, alive, rtrace, atrace)."""
    B = env.n_envs
    rt = torch.full((k, B), SENTINEL, dtype=torch.int32, device="cuda")
    at = torch.full((k, B), SENTINEL, dtype=torch.int32, device="cuda")
    obs, rew, steps = env.run(k, want_alive=True, reward_trace=rt, alive_trace=at, **kw)
    torch.cuda.synchronize()
    return (steps.cpu().numpy(), env.get_state().cpu().numpy(), obs.cpu().numpy(), rew.cpu().numpy(),
            env.last_alive().cpu().numpy(), rt.cpu().numpy(), at.cpu().numpy())


@pytest.mark.parametrize("side", FUSED + GENERIC)
@pytest.mark.parametrize("rule", list(RULES))
def test_period_1_equals_until_fixed(cuda, side, rule):
    rs = np.random.RandomState(side)
    B = 6
    cells = _soups(rs, B, side)
    cells[0] = 0                                            # fixed at step 1
    if side >= 4:
        cells[1] = place(side, BLOCK, 1, 1)
    for k in (1, 3, 4, 257):
        a, b = _env(cells, side, rule), _env(cells, side, rule)
        ref = _run(a, k, until_fixed=True)
        per = torch.full((B,), SENTINEL, dtype=torch.int32, device="cuda")
        got = _run(b, k, max_period=1, period_out=per)
        for x, y, name in zip(ref, got, ("steps", "world", "stable", "reward", "alive", "reward_trace", "alive_trace")):
            assert np.array_equal(x, y), (side, rule, k, name)
        steps, p = got[0], per.cpu().numpy()
        assert set(p.tolist()) <= {0, 1} and all(p[steps < k] == 1), (side, rule, k, p, steps)
        assert a.count == b.count == k


@pytest.mark.parametrize("c", CONVERGE, ids=lambda c: f"side{c['side']}-seed{c['seed']}")
def test_max_period_1_reproduces_reference_vectors(cuda, c):
    from cgl_b200.batched import BatchedSim
    env = BatchedSim(1, c["side"], seed=c["seed"], spawnStabilityFactor=c["spawn"], stableStabilityFactor=c["stable"])
    obs, rew, steps = env.run(c["limit"] + 1, want_alive=True, max_period=1)
    assert int(steps.item()) == c["steps"]
    assert int(rew.item()) == c["reward"] and int(env.last_alive().item()) == c["alive"]
    assert hashlib.sha256(env.get_state().cpu().numpy().tobytes()).hexdigest() == c["world_sha"]
    assert hashlib.sha256(obs.cpu().numpy().tobytes()).hexdigest() == c["stable_sha"]


def _mixed_batch(side, seed, n=37):
    """Empty, block, blinker, pulsar, figure eight, glider, a period-3 board (pulsar, shifted) and random soups."""
    rs = np.random.RandomState(seed)
    cells = _soups(rs, n, side)
    fixed = [np.zeros(side * side, np.uint8), place(side, BLOCK, 5, 7), place(side, BLINKER, 9, 3),
             place(side, PULSAR, 1, 2), place(side, FIGURE_EIGHT, 11, 13), place(side, GLIDER, 4, 4),
             place(side, PULSAR, 10, 6)]
    for i, w in enumerate(fixed):
        cells[(5 * i) % n] = w
    return cells


@pytest.mark.parametrize("P", [1, 2, 3, 8])
@pytest.mark.parametrize("rule", list(RULES))
@pytest.mark.parametrize("side,k", [(32, 127), (32, 300), (17, 200), (64, 150)])
def test_mixed_batch_matches_oracle_env_by_env(cuda, side, k, rule, P):
    spawn, smax, empty, emin = FACTORS
    cells = _mixed_batch(side, seed=side + P)
    B = len(cells)
    env = _env(cells, side, rule)
    st0 = env.stable.cpu().numpy().copy()
    per = torch.full((B,), SENTINEL, dtype=torch.int32, device="cuda")
    steps, world, stable, rew, alive, rt, at = _run(env, k, max_period=P, period_out=per)
    per = per.cpu().numpy()
    trips = set()
    for e in range(B):
        w, s = cells[e].copy(), st0[e].copy()
        rows = []
        t, p = run_cycle(w, s, side, spawn, smax, k, P, RULES[rule], empty, emin,
                         on_step=lambda t, ww, ss: rows.append((int(oracle.reward(ss)), int(oracle.alive(ww)))))
        what = (side, k, rule, P, e)
        assert (steps[e], per[e]) == (t, p), what
        assert np.array_equal(world[e], w) and np.array_equal(stable[e], s), what
        assert rew[e] == int(oracle.reward(s)) and alive[e] == int(oracle.alive(w)), what
        assert [tuple(r) for r in np.stack([rt[:t, e], at[:t, e]], 1).tolist()] == rows, what
        assert (rt[t:, e] == SENTINEL).all() and (at[t:, e] == SENTINEL).all(), what
        trips.add(t)
    assert len(trips) >= 3                                  # a CTA (or warp group) holds envs of different trip counts
    glider = 5 * 5 % B
    assert per[glider] == 0 and steps[glider] == k          # a spaceship is never a world cycle within 4*side steps
    if P == 2:
        assert per[6 * 5 % B] == 0 and steps[6 * 5 % B] == k      # period 3 under P = 2: the whole budget


@pytest.mark.parametrize("side", [12, 32, 64, 128, 100])
def test_a_match_at_the_last_step_counts(cuda, side):
    cells = np.stack([place(side, FIGURE_EIGHT)] * 3)       # period 8 from its first phase: world_8 == world_0
    for k, want in ((8, (8, 8)), (7, (7, 0))):
        env = _env(cells, side, "zero")
        per = torch.full((3,), SENTINEL, dtype=torch.int32, device="cuda")
        _, _, steps = env.run(k, max_period=8, period_out=per)
        assert steps.tolist() == [want[0]] * 3 and per.tolist() == [want[1]] * 3, (side, k)


@pytest.mark.parametrize("P,side", [(1, 268), (8, 237)])
def test_generic_side_at_the_bound(cuda, P, side):
    from cgl_b200 import native
    rs = np.random.RandomState(side)
    cells = _soups(rs, 2, side)
    cells[1] = place(side, PULSAR, 40, 50)
    env = _env(cells, side, "decay")
    st0 = env.stable.cpu().numpy().copy()
    per = torch.zeros(2, dtype=torch.int32, device="cuda")
    k = 40
    _, _, steps = env.run(k, max_period=P, period_out=per)
    spawn, smax, empty, emin = FACTORS
    for e in range(2):
        w, s = cells[e].copy(), st0[e].copy()
        t, p = run_cycle(w, s, side, spawn, smax, k, P, oracle.DEAD_DECAY, empty, emin)
        assert (int(steps[e]), int(per[e])) == (t, p)
        assert np.array_equal(env.get_state()[e].cpu().numpy(), w) and np.array_equal(env.stable[e].cpu().numpy(), s)
    if P == 8:
        assert int(per[1]) == 3
    from cgl_b200.batched import BatchedSim
    env2 = BatchedSim(1, side + 1, rng="device")
    with pytest.raises(native.CglNativeError, match="220 KiB"):
        env2.run(3, max_period=P)


def test_results_do_not_depend_on_cgl_run_impl(cuda):
    """CGL_RUN_IMPL picks the kernel of plain runs only; cycle runs give the same results with either value."""
    code = ("import sys, numpy as np, torch; sys.path[:0] = %r; import test_gpu_env_run_cycle as t; "
            "out = []\n"
            "for side in (32, 128, 17):\n"
            "    for P in (1, 2, 8):\n"
            "        env = t._env(t._mixed_batch(side, 3), side, 'decay')\n"
            "        per = torch.zeros(env.n_envs, dtype=torch.int32, device='cuda')\n"
            "        r = t._run(env, 100, max_period=P, period_out=per)\n"
            "        out.append(np.concatenate([x.astype(np.int64).ravel() for x in r] + [per.cpu().numpy()]))\n"
            "np.save(sys.argv[1], np.concatenate(out))\n") % ([HERE, os.path.dirname(HERE),
                                                             os.path.join(os.path.dirname(HERE), "ecen743-project-cgol_b200")],)
    import tempfile
    res = []
    with tempfile.TemporaryDirectory() as d:
        for impl in (None, "bytes", "sliced"):
            env = dict(os.environ)
            env.pop("CGL_RUN_IMPL", None)
            if impl:
                env["CGL_RUN_IMPL"] = impl
            path = os.path.join(d, f"{impl}.npy")
            r = subprocess.run([sys.executable, "-c", code, path], capture_output=True, text=True, env=env, timeout=600)
            assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
            res.append(np.load(path))
    assert np.array_equal(res[0], res[1]) and np.array_equal(res[0], res[2])


def test_ext_env_run_ex_max_period(cuda):
    from cgl_b200 import native
    ext = native.ext()
    side, B, k = 32, 5, 60
    cells = _mixed_batch(side, 1, B)
    a, b = _env(cells, side, "zero"), _env(cells, side, "zero")
    per = torch.zeros(B, dtype=torch.int32, device="cuda")
    steps = ext.env_run_ex(a._wa, a.stable, side, k, spawn=a.spawn, stable_max=a.stable_max, dead_rule=0, empty=0,
                           empty_min=-128, max_period=3, period=per)
    per_b = torch.zeros(B, dtype=torch.int32, device="cuda")
    _, _, steps_b = b.run(k, max_period=3, period_out=per_b)
    assert torch.equal(steps, steps_b) and torch.equal(per, per_b)
    assert torch.equal(a._wa, b._wa) and torch.equal(a.stable, b.stable)
    for kw in (dict(max_period=9), dict(max_period=-1), dict(max_period=2, until_fixed=True),
               dict(max_period=2, actions=torch.zeros((k, B), dtype=torch.int32, device="cuda")),
               dict(max_period=2, obs_trace=torch.zeros((k, B, side * side), dtype=torch.int8, device="cuda")),
               dict(max_period=0, period=per), dict(max_period=2, period=per[:3]),
               dict(max_period=2, period=per.to(torch.int64))):
        with pytest.raises(RuntimeError):
            ext.env_run_ex(a._wa, a.stable, side, k, **kw)


def test_batched_run_argument_errors(cuda):
    env = _env(_mixed_batch(32, 2, 4), 32, "zero")
    per = torch.zeros(4, dtype=torch.int32, device="cuda")
    for kw in (dict(max_period=9), dict(max_period=-1), dict(max_period=2.0), dict(max_period=2, until_fixed=True),
               dict(max_period=2, actions=torch.zeros((5, 4), dtype=torch.int32, device="cuda")),
               dict(max_period=2, obs_trace=torch.zeros((5, 4, 1024), dtype=torch.int8, device="cuda")),
               dict(period_out=per)):
        with pytest.raises(ValueError):
            env.run(5, **kw)
    for bad in (per.cpu(), per.to(torch.int64), per[:3], torch.zeros((4, 2), dtype=torch.int32, device="cuda")[:, 0],
                [0, 0, 0, 0]):
        with pytest.raises(TypeError):
            env.run(5, max_period=2, period_out=bad)
    assert env.count == 0


@pytest.mark.parametrize("fork", [False, True])
def test_facade_run_until_cycle(cuda, fork):
    import importlib.util
    if fork:
        spec = importlib.util.spec_from_file_location(
            "CGL_fork", os.path.join(os.path.dirname(HERE), "ecen743-project-cgol_b200", "CGL_action+", "CGL.py"))
        CGL = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(CGL)
        kw = dict(empty=-1, empty_min=-5)
        rule, empty, emin = oracle.DEAD_DECAY, -1, -5
    else:
        import CGL
        kw, rule, empty, emin = {}, oracle.DEAD_ZERO, 0, -128
    side, spawn, smax = 20, -2, 2
    env = CGL.sim(side=side, seed=4, gpu=True, spawnStabilityFactor=spawn, stableStabilityFactor=smax, **kw)
    w = env.get_state(vector=True).astype(np.uint8).copy()
    s = env.get_stable(vector=True).astype(np.int8).copy()
    env.toggle_state(np.int32(33))                          # pending: applied before the run, as before step()
    (oracle.toggle_masked if fork else oracle.toggle)(w, s, 33, spawn)
    n, p = env.run_until_cycle(2000, max_period=2)
    t, q = run_cycle(w, s, side, spawn, smax, 2000, 2, rule, empty, emin)
    assert (n, p) == (t, q) and env.get_count() == n
    assert np.array_equal(env.get_state(vector=True), w) and np.array_equal(env.get_stable(vector=True), s)
    assert int(env.reward()) == int(oracle.reward(s))
    n2, p2 = env.run_until_cycle(50, max_period=8)          # already in its cycle: stops within one period
    assert 1 <= n2 == p2 <= 8 or (p2 == 0 and n2 == 50)
    assert env.get_count() == n + n2
