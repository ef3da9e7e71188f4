"""GPU suite: everything that waits on the device (chained env steps, chained life strips) and the
one-launch facade step -- ordering, boundedness and "no result computed from stale data".

Round-2 regression tests for the advisor's findings:
  * chained env steps with THREE or more launches queued / captured in one graph on small batches (three grids
    fit on the GPU at once): a two-valued plane token is only sound because a CTA lets its dependents launch
    after its own wait succeeded (csrc/cgl_env.cu);
  * a token that never arrives raises an error and leaves the state untouched instead of stepping stale planes;
  * back-to-back toggle_state + step pairs on the facade without any read in between (the action travels by
    value, cgl_sim_step) -- reference semantics: CGL/CGL.py:322-328 applies each toggle immediately.
"""
import ctypes

import numpy as np
import pytest

from oracle import oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SPAWN, STABLE = -2, 2


@pytest.fixture(scope="module")
def B():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200.batched import BatchedSim
    return BatchedSim


@pytest.fixture(scope="module")
def native(B):
    from cgl_b200 import native as n
    return n


def host_state(env):
    return env.get_state().cpu().numpy(), env.stable.cpu().numpy().copy()


@pytest.mark.parametrize("side", [32, 64, 128])
@pytest.mark.parametrize("n_envs", [1, 8, 64])
def test_graph_of_eight_chained_steps_matches_oracle(B, side, n_envs, monkeypatch):
    monkeypatch.setenv("CGL_ENV_CHAINED", "1")
    env = B(n_envs, side, seed=11, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
    assert env.chained
    cells, st = host_state(env)
    size = side * side
    rs = np.random.RandomState(side + n_envs)
    acts_h = rs.randint(size + 1, size=(8, n_envs)).astype(np.int32)
    acts = torch.from_numpy(acts_h).cuda()
    env.step(acts[0]); env.step(acts[1])                    # warm-up outside the capture (2 steps: planes back in place)
    for t in range(2):
        oracle.step_batch(cells, st, side, acts_h[t], SPAWN, STABLE, threads=2)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            for t in range(8):
                env.step(acts[t])
    replays = 3
    for _ in range(replays):
        graph.replay()
    torch.cuda.synchronize()
    rew_o = None
    for _ in range(replays):
        for t in range(8):
            rew_o, _ = oracle.step_batch(cells, st, side, acts_h[t], SPAWN, STABLE, threads=2)
    w, s = host_state(env)
    assert np.array_equal(w, cells) and np.array_equal(s, st)
    assert np.array_equal(env._reward.cpu().numpy(), rew_o)
    env.check_actions()


@pytest.mark.parametrize("n_envs", [1, 5, 64, 300])
def test_many_queued_chained_steps_match_oracle(B, n_envs, monkeypatch):
    """A backed-up stream: 40 chained launches enqueued without any synchronisation in between."""
    monkeypatch.setenv("CGL_ENV_CHAINED", "1")
    side, size = 64, 64 * 64
    env = B(n_envs, side, seed=3, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
    cells, st = host_state(env)
    rs = np.random.RandomState(n_envs)
    acts_h = rs.randint(size + 1, size=(40, n_envs)).astype(np.int32)
    acts = torch.from_numpy(acts_h).cuda()
    blocker = torch.empty(1 << 28, dtype=torch.uint8, device="cuda")
    for _ in range(4):
        blocker.fill_(1)                                    # keep the GPU busy while the launches pile up
    for t in range(40):
        _, rew, _ = env.step(acts[t])
    torch.cuda.synchronize()
    for t in range(40):
        rew_o, _ = oracle.step_batch(cells, st, side, acts_h[t], SPAWN, STABLE, threads=2)
    w, s = host_state(env)
    assert np.array_equal(w, cells) and np.array_equal(s, st) and np.array_equal(rew.cpu().numpy(), rew_o)


def test_stale_env_token_raises_and_leaves_state_untouched(B, native):
    lib = native.load()
    side, n = 64, 6
    env = B(n, side, seed=5, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
    cells, st = host_state(env)
    wa_before = env._wa.clone()
    tokens = torch.full((n,), 1, dtype=torch.int32, device="cuda")
    tokens[2] = 7                                           # env 2's predecessor "never ran"
    reward = torch.full((n,), -12345, dtype=torch.int32, device="cuda")
    alarm = native.alarm()
    alarm[:] = 0
    native.check(lib.cgl_set_wait_timeout_ms(100))
    try:
        native.check(lib.cgl_env_step_chained(native.dptr(env._wa), native.dptr(env._wb), native.dptr(env.stable), n,
                                              side, None, SPAWN, STABLE, native.dptr(reward), None,
                                              native.dptr(env._err), native.dptr(tokens), 1, 2,
                                              native.current_stream()))
        torch.cuda.synchronize()
    finally:
        native.check(lib.cgl_set_wait_timeout_ms(2000))
    assert alarm[1] == 1
    with pytest.raises(native.CglNativeError):
        native.check_alarm()
    assert alarm[1] == 0
    with pytest.raises(native.CglNativeError):
        env.check_actions()
    # env 2: nothing written, token not published; every other env stepped normally
    out = torch.empty((n, side * side), dtype=torch.uint8, device="cuda")
    native.check(lib.cgl_unpack(native.dptr(env._wb), native.dptr(out), n, side, side, native.current_stream()))
    w_new, s_new, tok = out.cpu().numpy(), env.stable.cpu().numpy(), tokens.cpu().numpy()
    assert torch.equal(env._wa, wa_before)
    for e in range(n):
        if e == 2:
            assert np.array_equal(s_new[e], st[e]) and tok[e] == 7 and int(reward[e]) == -12345
        else:
            oracle.step(cells[e], st[e], side, SPAWN, STABLE)
            assert np.array_equal(w_new[e], cells[e]) and np.array_equal(s_new[e], st[e]) and tok[e] == 2
            assert int(reward[e]) == int(oracle.reward(st[e]))


def test_stale_life_token_raises_and_stores_nothing(native):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    lib = native.load()
    rows, cols = 512, 32 * 64
    a = torch.randint(-2 ** 31, 2 ** 31 - 1, (rows * cols // 32,), dtype=torch.int32, device="cuda")
    b = torch.full_like(a, 0x5A5A5A5A)
    a0 = a.clone()
    alarm = native.alarm()
    alarm[:] = 0
    res = ctypes.c_int(-1)
    native.check(lib.cgl_set_wait_timeout_ms(100))
    try:
        native.check(lib.cgl_test_fault(1))
        native.check(lib.cgl_life_run(native.dptr(a), native.dptr(b), rows, cols, 1, 8, 8, ctypes.byref(res),
                                      native.current_stream()))
        torch.cuda.synchronize()
    finally:
        native.check(lib.cgl_set_wait_timeout_ms(2000))
    assert alarm[2] == 1
    with pytest.raises(native.CglNativeError):
        native.check_alarm()
    assert torch.equal(a, a0) and bool((b == 0x5A5A5A5A).all())      # no strip stored anything
    # and the next run is healthy again
    native.check(lib.cgl_life_run(native.dptr(a), native.dptr(b), rows, cols, 1, 8, 8, ctypes.byref(res),
                                  native.current_stream()))
    torch.cuda.synchronize()
    native.check_alarm()
    assert not bool((b == 0x5A5A5A5A).all())


@pytest.mark.parametrize("side", [10, 64, 128, 200])
def test_facade_toggle_step_pairs_without_reads(side):
    """toggle_state(a); step(); toggle_state(b); step() with no observation in between, right behind a long
    deferred run that keeps the stream busy: each step must apply ITS toggle (the action travels by value)."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import CGL
    size = side * side
    env = CGL.sim(side=side, seed=2, gpu=True, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
    ref = oracle.OracleSim(side=side, seed=2, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
    n_plain = 3000 if side <= 128 else 300
    for _ in range(n_plain):
        env.step()
        ref.step()
    rs = np.random.RandomState(side)
    acts = rs.randint(size, size=12)
    for a in acts:
        env.toggle_state(np.int32(a)); env.step()
        ref.toggle_state(np.int32(a)); ref.step()
    assert int(env.reward()) == int(ref.reward()) and int(env.alive()) == int(ref.alive())
    assert np.array_equal(env.get_state(vector=True), ref.world)
    assert np.array_equal(env.get_stable(vector=True), ref.stable)
    assert env.get_count() == n_plain + 12


@pytest.mark.parametrize("side", [5, 10, 33, 64, 100, 320, 448])
def test_sim_step_one_launch_matches_oracle(side, native):
    """cgl_sim_step through the C ABI: mirror, reward, live count and sequence word, base and fork rules."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    lib = native.load()
    size, W = side * side, (side + 31) // 32
    rs = np.random.RandomState(side)
    for rule, empty, emin, masked in ((0, 0, 0, 0), (1, -1, -6, 1), (2, -1, -6, 1)):
        cells = rs.randint(2, size=size).astype(np.uint8)
        st = rs.randint(-128, 128, size=size).astype(np.int8)
        wa = torch.zeros(side * W, dtype=torch.int32, device="cuda")
        wb = torch.zeros_like(wa)
        c_d = torch.from_numpy(cells).cuda()
        s_d = torch.from_numpy(st.copy()).cuda()
        native.check(lib.cgl_pack(native.dptr(c_d), native.dptr(wa), 1, side, side, native.current_stream()))
        mirror = torch.zeros(size, dtype=torch.int8).pin_memory()
        res = torch.zeros(4, dtype=torch.int32).pin_memory()
        for t in range(6):
            a = int(rs.randint(size + 1))
            native.check(lib.cgl_sim_step(native.dptr(wa), native.dptr(wb), native.dptr(s_d), side, a, SPAWN, STABLE,
                                          rule, empty, emin, masked, native.dptr(mirror), native.dptr(res), t + 1,
                                          native.current_stream()))
            wa, wb = wb, wa
            torch.cuda.synchronize()
            if a < size:
                (oracle.toggle_masked if masked else oracle.toggle)(cells, st, a, SPAWN)
            oracle.step_rule(cells, st, side, SPAWN, STABLE, rule, empty, emin)
            native.check(lib.cgl_unpack(native.dptr(wa), native.dptr(c_d), 1, side, side, native.current_stream()))
            assert np.array_equal(c_d.cpu().numpy(), cells), (side, rule, t)
            assert np.array_equal(s_d.cpu().numpy(), st) and np.array_equal(mirror.numpy(), st), (side, rule, t)
            assert int(res[0]) == int(oracle.reward(st)) and int(res[1]) == int(oracle.alive(cells)) and int(res[2]) == t + 1


def test_sim_step_rejects_side_above_limit(native):
    """448 is the largest side whose byte plane and packed next world fit in shared memory; 449 is refused before any
    launch."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    lib = native.load()
    side = 449
    wa = torch.zeros(side * ((side + 31) // 32), dtype=torch.int32, device="cuda")
    wb = torch.zeros_like(wa)
    s_d = torch.zeros(side * side, dtype=torch.int8, device="cuda")
    with pytest.raises(native.CglNativeError, match="side must be <= 448"):
        native.check(lib.cgl_sim_step(native.dptr(wa), native.dptr(wb), native.dptr(s_d), side, side * side, SPAWN, STABLE,
                                      0, 0, 0, 0, None, None, 1, native.current_stream()))
