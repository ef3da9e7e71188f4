"""BatchedSim.run(k, until_settled=True) and the facades' run_until_settled (cgl_env_run_settle) on the GPU.

  * mixed batches (still lifes, oscillators up to period 15, a lone glider and a lightweight spaceship, a glider that
    hits a block, reference soups) agree env by env with a brute force that keeps every past world, in steps,
    period, world, plane, reward, alive and trace rows, on fused and generic sides, all three dead-cell rules, with
    and without traces, trace rows from steps[e] on untouched;
  * every env with period <= 8 equals run(k, max_period=8), and every env equals a plain run(steps[e]);
  * the budget edges: a match exactly at max_steps, mu + lambda = max_steps + 1, a glider at 256^2 (period 1024) and
    max_steps = 2^32 - 1;
  * the torch extension, BatchedSim's argument errors and run_until_settled on both facades."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from oracle_settle import run_settle

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
RULES = {"zero": oracle.DEAD_ZERO, "decay": oracle.DEAD_DECAY, "sat": oracle.DEAD_SAT}
FACTORS = (-2, 2, -1, -5)                     # spawn, stable_max, empty, empty_min
SENTINEL = -12345

BLOCK = [(0, 0), (0, 1), (1, 0), (1, 1)]
BLINKER = [(0, 0), (0, 1), (0, 2)]
PULSAR = [rc for r in (0, 5, 7, 12) for c in (2, 3, 4, 8, 9, 10) for rc in ((r, c), (c, r))]          # period 3
FIGURE_EIGHT = [(r, c) for r in range(3) for c in range(3)] + [(r + 3, c + 3) for r in range(3) for c in range(3)]
PENTADECATHLON = [(r, 1) for r in (0, 1, 3, 4, 5, 6, 8, 9)] + [(2, 0), (2, 2), (7, 0), (7, 2)]            # period 15
GLIDER = [(0, 1), (1, 2), (2, 0), (2, 1), (2, 2)]                  # moves down-right: period 4*side on a torus
LWSS = [(0, 1), (0, 4), (1, 0), (2, 0), (2, 4), (3, 0), (3, 1), (3, 2), (3, 3)]   # period 2*side (even), 4*side (odd)


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


def _run(env, k, traced=True, **kw):
    """run(k, ...) with sentinel-filled traces; returns (steps, world, stable, reward, alive, rtrace, atrace)."""
    B = env.n_envs
    rt = torch.full((k, B), SENTINEL, dtype=torch.int32, device="cuda") if traced else None
    at = torch.full((k, B), SENTINEL, dtype=torch.int32, device="cuda") if traced else None
    obs, rew, steps = env.run(k, want_alive=True, reward_trace=rt, alive_trace=at, **kw)
    torch.cuda.synchronize()
    return (steps.cpu().numpy(), env.get_state().cpu().numpy(), obs.cpu().numpy(), rew.cpu().numpy(),
            env.last_alive().cpu().numpy(), None if rt is None else rt.cpu().numpy(),
            None if at is None else at.cpu().numpy())


def brute_force(world, stable, side, k, rule, on_step=None):
    """Steps one env in place, every past world in a dict; (t, p) at the first world seen before, or (k, 0)."""
    spawn, smax, empty, emin = FACTORS
    seen = {np.packbits(world).tobytes(): 0}
    for t in range(1, k + 1):
        oracle.step_rule(world, stable, side, spawn, smax, RULES[rule], empty, emin)
        if on_step is not None:
            on_step(t, world, stable)
        key = np.packbits(world).tobytes()
        if key in seen:
            return t, t - seen[key]
        seen[key] = t
    return k, 0


def _mixed_batch(side, seed, n=23):
    """Known boards where they fit, reference soups (seeded as the reference seeds its worlds) elsewhere."""
    cells = np.stack([oracle.initial_world(side, 100 * seed + i) for i in range(n)])
    fixed = [np.zeros(side * side, np.uint8), place(side, BLOCK, 5, 7), place(side, BLINKER, 9, 3),
             place(side, PULSAR, 1, 2), place(side, FIGURE_EIGHT, 11, 13), place(side, PENTADECATHLON, 3, 9),
             place(side, GLIDER, 4, 4), place(side, LWSS, 6, 1)]
    if side >= 32:
        fixed.append(place(side, GLIDER, 0, 0) | place(side, BLOCK, 14, 15))     # mu > 0 with a long lambda
    for i, w in enumerate(fixed):
        cells[(3 * i) % n] = w
    return cells


FUSED_K = [(32, 200), (64, 300), (96, 420), (128, 560), (256, 1070)]
GENERIC_K = [(1, 5), (2, 9), (3, 20), (17, 90), (33, 160), (100, 420), (200, 820)]


@pytest.mark.parametrize("traced", [True, False])
@pytest.mark.parametrize("side,k,rule", [(s, k, r) for s, k in FUSED_K[:1] + GENERIC_K[3:4] for r in RULES] +
                         [(s, k, list(RULES)[i % 3]) for i, (s, k) in enumerate(FUSED_K[1:] + GENERIC_K[:3] +
                                                                                  GENERIC_K[4:])])
def test_mixed_batch_matches_brute_force_env_by_env(cuda, side, k, rule, traced):
    cells = _mixed_batch(side, seed=side)
    B = len(cells)
    env = _env(cells, side, rule)
    st0 = env.stable.cpu().numpy().copy()
    per = torch.full((B,), SENTINEL, dtype=torch.int32, device="cuda")
    steps, world, stable, rew, alive, rt, at = _run(env, k, traced, until_settled=True, period_out=per)
    per = per.cpu().numpy()
    for e in range(B):
        w, s = cells[e].copy(), st0[e].copy()
        rows = []
        t, p = brute_force(w, s, side, k, rule,
                           on_step=lambda t, ww, ss: rows.append((int(oracle.reward(ss)), int(oracle.alive(ww)))))
        what = (side, k, rule, e)
        assert (steps[e], per[e]) == (t, p), what
        assert np.array_equal(world[e], w) and np.array_equal(stable[e], s), what
        assert rew[e] == int(oracle.reward(s)) and alive[e] == int(oracle.alive(w)), what
        if traced:
            assert [tuple(r) for r in np.stack([rt[:t, e], at[:t, e]], 1).tolist()] == rows, what
            assert (rt[t:, e] == SENTINEL).all() and (at[t:, e] == SENTINEL).all(), what
    if side >= 32:
        assert (steps[18], per[18]) == (4 * side, 4 * side)          # the lone glider
        lw = (2 if side % 2 == 0 else 4) * side
        assert (steps[21], per[21]) == (lw, lw)                      # the lightweight spaceship
        assert per[15] == 15 and per[9] == 3 and per[12] == 8       # pentadecathlon, pulsar, figure eight
        assert per[1] == 0 or steps[1] > per[1]                      # the glider that hits a block: mu > 0
    assert env.count == k


@pytest.mark.parametrize("side,k", [(32, 200), (64, 300), (128, 560), (17, 90), (100, 420)])
def test_short_periods_equal_max_period_8_and_every_env_a_plain_run(cuda, side, k):
    cells = _mixed_batch(side, seed=side + 1)
    B = len(cells)
    a, b = _env(cells, side, "decay"), _env(cells, side, "decay")
    pa = torch.zeros(B, dtype=torch.int32, device="cuda")
    pb = torch.zeros(B, dtype=torch.int32, device="cuda")
    ra = _run(a, k, until_settled=True, period_out=pa)
    rb = _run(b, k, max_period=8, period_out=pb)
    pa, pb = pa.cpu().numpy(), pb.cpu().numpy()
    short = (pa >= 1) & (pa <= 8)
    assert short.sum() >= 4
    assert np.array_equal(pa[short], pb[short])
    for x, y, name in zip(ra, rb, ("steps", "world", "stable", "reward", "alive", "reward_trace", "alive_trace")):
        assert np.array_equal(x[..., short], y[..., short]) if name.endswith("trace") else \
            np.array_equal(x[short], y[short]), name
    for e in range(B):                               # a plain run of steps[e] leaves the same state
        c = _env(cells[e:e + 1], side, "decay")
        obs, rew, _ = c.run(int(ra[0][e]), want_alive=True)
        assert np.array_equal(c.get_state().cpu().numpy()[0], ra[1][e]), e
        assert np.array_equal(obs.cpu().numpy()[0], ra[2][e]), e
        assert int(rew[0]) == ra[3][e] and int(c.last_alive()[0]) == ra[4][e], e


@pytest.mark.parametrize("side", [32, 64, 12, 100])
def test_budget_edges(cuda, side):
    per = torch.zeros(3, dtype=torch.int32, device="cuda")
    # a match exactly at max_steps counts; one step less is no match
    cells = np.stack([place(side, FIGURE_EIGHT)] * 2 + [place(side, GLIDER)])
    for k, want in ((8, [(8, 8), (8, 8), (8, 0)]), (7, [(7, 0)] * 3)):
        env = _env(cells, side, "zero")
        _, _, steps = env.run(k, until_settled=True, period_out=per)
        assert list(zip(steps.tolist(), per.tolist())) == want, (side, k)
    for k, want in ((4 * side, (4 * side, 4 * side)), (4 * side - 1, (4 * side - 1, 0))):
        env = _env(cells[2:], side, "zero")
        p1 = torch.zeros(1, dtype=torch.int32, device="cuda")
        _, _, steps = env.run(k, until_settled=True, period_out=p1)
        assert (int(steps[0]), int(p1[0])) == want, (side, k)
    # mu + lambda = max_steps + 1: reports (max_steps, 0) and runs max_steps steps
    rs = np.random.RandomState(side)
    soups = (rs.random_sample((4, side * side)) < 0.35).astype(np.uint8)
    for e in range(4):
        T, lam = brute_force(soups[e].copy(), np.zeros(side * side, np.int8), side, 20000, "zero")
        assert lam > 0
        for M, want in ((T, (T, lam)), (T - 1, (T - 1, 0))):
            env = _env(soups[e:e + 1], side, "sat")
            w, s = soups[e].copy(), env.stable.cpu().numpy()[0].copy()
            p1 = torch.zeros(1, dtype=torch.int32, device="cuda")
            obs, rew, steps = env.run(M, until_settled=True, period_out=p1)
            assert (int(steps[0]), int(p1[0])) == want, (side, e, M)
            spawn, smax, empty, emin = FACTORS
            for _ in range(want[0]):
                oracle.step_rule(w, s, side, spawn, smax, oracle.DEAD_SAT, empty, emin)
            assert np.array_equal(env.get_state().cpu().numpy()[0], w) and np.array_equal(obs.cpu().numpy()[0], s)


def test_glider_at_256_has_period_1024(cuda):
    cells = np.stack([place(256, GLIDER, 7, 200), place(256, LWSS, 100, 3), place(256, BLOCK)])
    env = _env(cells, 256, "decay")
    per = torch.zeros(3, dtype=torch.int32, device="cuda")
    _, _, steps = env.run(1200, until_settled=True, period_out=per)
    assert steps.tolist() == [1024, 512, 1] and per.tolist() == [1024, 512, 1]
    env = _env(cells, 256, "decay")
    _, _, steps = env.run(1023, until_settled=True, period_out=per)
    assert steps.tolist() == [1023, 512, 1] and per.tolist() == [0, 512, 1]


@pytest.mark.parametrize("side", [32, 128, 17])
def test_the_largest_budget_stops_at_the_settle_time(cuda, side):
    """max_steps = 2^32 - 1: 2 * max_steps passes 2^32, and boards that settle stop there."""
    cells = np.stack([np.zeros(side * side, np.uint8), place(side, BLOCK), place(side, BLINKER, 5, 5),
                      place(side, GLIDER), place(side, FIGURE_EIGHT, 1, 1)])
    env = _env(cells, side, "zero")
    st0 = env.stable.cpu().numpy().copy()
    per = torch.zeros(len(cells), dtype=torch.int32, device="cuda")
    _, _, steps = env.run(2 ** 32 - 1, until_settled=True, period_out=per)
    for e in range(len(cells)):
        w, s = cells[e].copy(), st0[e].copy()
        assert (int(steps[e]), int(per[e])) == brute_force(w, s, side, 10 * side, "zero"), e
        assert np.array_equal(env.get_state()[e].cpu().numpy(), w) and np.array_equal(env.stable[e].cpu().numpy(), s)
    assert env.count == 2 ** 32 - 1


def test_generic_side_at_the_bound(cuda):
    from cgl_b200 import native
    from cgl_b200.batched import BatchedSim
    side = 274
    cells = np.stack([oracle.initial_world(side, 5), place(side, GLIDER)])
    env = _env(cells, side, "decay")
    st0 = env.stable.cpu().numpy().copy()
    per = torch.zeros(2, dtype=torch.int32, device="cuda")
    _, _, steps = env.run(60, until_settled=True, period_out=per)
    spawn, smax, empty, emin = FACTORS
    for e in range(2):
        w, s = cells[e].copy(), st0[e].copy()
        t, p = run_settle(w, s, side, spawn, smax, 60, oracle.DEAD_DECAY, empty, emin)
        assert (int(steps[e]), int(per[e])) == (t, p)
        assert np.array_equal(env.get_state()[e].cpu().numpy(), w) and np.array_equal(env.stable[e].cpu().numpy(), s)
    env2 = BatchedSim(1, side + 1, rng="device")
    with pytest.raises(native.CglNativeError, match="side <= 274"):
        env2.run(3, until_settled=True)


def test_ext_env_run_ex_until_settled(cuda):
    from cgl_b200 import native
    ext = native.ext()
    side, B, k = 32, 9, 200
    cells = _mixed_batch(side, 1, B)
    a, b = _env(cells, side, "zero"), _env(cells, side, "zero")
    per = torch.zeros(B, dtype=torch.int32, device="cuda")
    steps = ext.env_run_ex(a._wa, a.stable, side, k, spawn=a.spawn, stable_max=a.stable_max, dead_rule=0, empty=0,
                           empty_min=-128, until_settled=True, period=per)
    per_b = torch.zeros(B, dtype=torch.int32, device="cuda")
    _, _, steps_b = b.run(k, until_settled=True, period_out=per_b)
    assert torch.equal(steps, steps_b) and torch.equal(per, per_b)
    assert torch.equal(a._wa, b._wa) and torch.equal(a.stable, b.stable)
    for kw in (dict(until_settled=True, max_period=2), dict(until_settled=True, until_fixed=True),
               dict(until_settled=True, actions=torch.zeros((k, B), dtype=torch.int32, device="cuda")),
               dict(until_settled=True, obs_trace=torch.zeros((k, B, side * side), dtype=torch.int8, device="cuda")),
               dict(until_settled=True, period=per[:3]), dict(until_settled=True, period=per.to(torch.int64)),
               dict(period=per)):
        with pytest.raises(RuntimeError):
            ext.env_run_ex(a._wa, a.stable, side, k, **kw)


def test_batched_run_argument_errors(cuda):
    env = _env(_mixed_batch(32, 2, 4), 32, "zero")
    per = torch.zeros(4, dtype=torch.int32, device="cuda")
    for kw in (dict(until_settled=True, max_period=2), dict(until_settled=True, until_fixed=True),
               dict(until_settled=True, actions=torch.zeros((5, 4), dtype=torch.int32, device="cuda")),
               dict(until_settled=True, obs_trace=torch.zeros((5, 4, 1024), dtype=torch.int8, device="cuda"))):
        with pytest.raises(ValueError):
            env.run(5, **kw)
    with pytest.raises(ValueError, match="period_out needs max_period"):
        env.run(5, period_out=per)
    for bad in (per.cpu(), per.to(torch.int64), per[:3], torch.zeros((4, 2), dtype=torch.int32, device="cuda")[:, 0],
                [0, 0, 0, 0]):
        with pytest.raises(TypeError):
            env.run(5, until_settled=True, period_out=bad)
    assert env.count == 0
    _, _, steps = env.run(5, until_settled=True)                # period_out is optional
    assert env.count == 5 and steps.shape == (4,)


@pytest.mark.parametrize("fork", [False, True])
def test_facade_run_until_settled(cuda, fork):
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
    toggle = oracle.toggle_masked if fork else oracle.toggle
    env.toggle_state(np.int32(33))                          # deferred: applied before the run, as before step()
    toggle(w, s, 33, spawn)
    env.step()
    oracle.step_rule(w, s, side, spawn, smax, rule, empty, emin)
    env.toggle_state(np.int32(150))
    toggle(w, s, 150, spawn)
    n, p = env.run_until_settled(5000)
    t, q = run_settle(w, s, side, spawn, smax, 5000, rule, empty, emin)
    assert (n, p) == (t, q) and p > 0 and env.get_count() == 1 + n
    assert np.array_equal(env.get_state(vector=True), w) and np.array_equal(env.get_stable(vector=True), s)
    assert int(env.reward()) == int(oracle.reward(s))
    n2, p2 = env.run_until_settled(50)                      # already in its cycle: stops after one period
    assert n2 == p2 == p or (p2 == 0 and n2 == 50 and p > 50)
    assert env.get_count() == 1 + n + n2
