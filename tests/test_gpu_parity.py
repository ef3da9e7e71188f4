"""GPU suite (-m gpu): the CUDA path, called through the C ABI (libcgl_b200.so), against
 (a) the golden vectors recorded from the reference's own CPU step (tests/golden/), and
 (b) the CPU oracle on the same seeded inputs, bit-exact (all arithmetic is integer).
Nothing here reads /root/reference."""
import json
import os

import numpy as np
import pytest

from conftest import ROOT, TRACES
from oracle import oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

API = json.load(open(os.path.join(ROOT, "tests", "golden", "golden_api.json")))


@pytest.fixture(scope="module")
def cgl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    os.environ.pop("GPU_CAPABLE", None)
    import importlib
    import CGL
    return importlib.reload(CGL)


@pytest.fixture(scope="module")
def B(cgl):
    from cgl_b200.batched import BatchedSim
    return BatchedSim


def dev_np(t):
    return t.detach().cpu().numpy()


# ------------------------------------------------------------------------------------------
# (a) golden traces through the reference-facing facade
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(TRACES))
def test_facade_replays_reference_trace(cgl, name):
    tr = TRACES[name]
    env = cgl.sim(state=tr.worlds[0].reshape(tr.side, tr.side), gpu=True,
                  spawnStabilityFactor=tr.spawn, stableStabilityFactor=tr.stable_max)
    assert np.array_equal(env.get_stable(vector=True), tr.stables[0])
    assert env.reward() == tr.rewards[0] and env.alive() == tr.alives[0]
    obs = env.get_stable(vector=True, shallow=True)
    for t in range(tr.T):
        a = tr.action(t)
        if a is not None:
            env.toggle_state(np.int32(a) if isinstance(a, int) else a)
        assert env.reward() == tr.rewards_after_toggle[t], (name, t)
        env.step()
        assert np.array_equal(env.get_state(vector=True), tr.worlds[t + 1]), (name, t)
        assert np.array_equal(env.get_stable(vector=True), tr.stables[t + 1]), (name, t)
        assert obs is env.get_stable(vector=True, shallow=True)           # N1 aliasing
        assert np.array_equal(obs, tr.stables[t + 1])
        r, al = env.reward(), env.alive()
        assert isinstance(r, np.int32) and isinstance(al, np.uint32)
        assert r == tr.rewards[t + 1] and al == tr.alives[t + 1]
    assert env.get_count() == tr.T


def test_facade_random_start_uses_reference_rng(cgl):
    tr = TRACES["rand64_plain"]
    env = cgl.sim(side=64, seed=0, gpu=True, spawnStabilityFactor=-2, stableStabilityFactor=2)
    assert np.array_equal(env.get_state(vector=True), tr.worlds[0])
    for t in range(10):
        env.step()
    assert np.array_equal(env.get_state(vector=True), tr.worlds[10])
    assert np.array_equal(env.get_stable(vector=True), tr.stables[10])
    assert (env.alive(), env.reward()) == (772, -691)                      # SURVEY.md 8c golden (3)


def test_facade_api_behaviour_matches_reference(cgl):
    w0 = np.array(API["side6_seed3_world"], np.uint8)
    env = cgl.sim(side=6, seed=3, gpu=True)
    assert np.array_equal(env.get_state(vector=True), w0)
    env.toggle_state([3, 3])
    assert (env.get_state(vector=True) != w0).sum() == 1                   # duplicates toggle once
    env.toggle_state(36)                                                   # "do nothing"
    assert (env.get_state(vector=True) != w0).sum() == 1
    env.toggle_state([36])
    for bad in (37, -1, [1, 99]):
        with pytest.raises(ValueError):
            env.toggle_state(bad)
    with pytest.raises(IndexError):
        env.toggle_state([])
    env = cgl.sim(side=5, seed=1, gpu=True, spawnStabilityFactor=-2, stableStabilityFactor=2)
    g = API["getters"]
    assert (env.get_side(), env.get_count(), env.get_seed(), env.get_state_dim(), str(env.get_state_space_dim()),
            env.get_action_space_dim()) == (g["side"], g["count"], g["seed"], g["state_dim"], g["state_space_dim"],
                                            g["action_space_dim"])
    init_w, init_s = env.get_state(vector=True), env.get_stable(vector=True)
    env.step(); env.step()
    assert env.get_count() == API["count_after_2"]
    env.reset()
    assert env.get_count() == API["count_after_reset"]
    assert np.array_equal(env.get_state(vector=True), init_w) and np.array_equal(env.get_stable(vector=True), init_s)
    with pytest.raises(ValueError):
        env.update_state(np.zeros(9), 3)
    with pytest.raises(ValueError):
        env.update_state(np.zeros(25), 4)
    new = np.arange(25) % 2
    env.update_state(new, 5)
    assert np.array_equal(env.get_state(vector=True), new) and np.array_equal(env.get_stable(vector=True), init_s)
    assert env.match(new.reshape(5, 5)) is True and env.match(1 - new) is False
    sv = env.save()
    assert len(sv) == 6 and [type(v).__name__ for v in sv] == API["save_types"]
    with pytest.raises(TypeError):
        env.load([1], np.zeros(1, np.int8), 1, 0, -1, 1)
    with pytest.raises(ValueError):
        env.load(np.zeros(1), np.zeros(1), 0, 0, -1, 1)
    with pytest.raises(ValueError):
        env.load(np.zeros(1), np.zeros(1), 1, -1, -1, 1)
    with pytest.raises(TypeError):
        env.load(np.zeros(1), np.zeros(1), 1, 0, -1.0, 1)
    # save -> step -> load restores; load with another side re-allocates
    env.step()
    env.load(*sv)
    assert np.array_equal(env.get_state(vector=True), sv[0]) and np.array_equal(env.get_stable(vector=True), sv[1])
    tr = TRACES["tiny7"]
    env.load(tr.worlds[2], tr.stables[2], 7, 2, tr.spawn, tr.stable_max)
    a = tr.action(2)
    env.toggle_state(a); env.step()
    assert np.array_equal(env.get_state(vector=True), tr.worlds[3]) and np.array_equal(env.get_stable(vector=True), tr.stables[3])
    assert env.get_state().shape == (7, 7) and env.get_stable().dtype == np.int8 and env.get_state().dtype == np.uint8
    with pytest.raises(RuntimeError):
        env.step(forceCPU=True)
    with pytest.raises(ValueError):
        cgl.sim(state=np.array([0, 2, 1, 0]), gpu=True)


# ------------------------------------------------------------------------------------------
# (b) batched driver vs golden envs and vs the oracle
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("side,n", [(64, 6), (128, 2)])
def test_batched_fused_matches_golden_envs(B, side, n):
    trs = [TRACES[f"env{side}_{e}"] for e in range(n)]
    env = B(n, side, seed=0, spawnStabilityFactor=-2, stableStabilityFactor=2)      # env e seeded seed+e
    assert env.fused
    assert np.array_equal(dev_np(env.get_state()), np.stack([t.worlds[0] for t in trs]))
    for t in range(trs[0].T):
        acts = torch.tensor([tr.actions[t, 0] for tr in trs], dtype=torch.int32, device="cuda")
        obs, rew, done = env.step(acts, want_alive=True)
        assert np.array_equal(dev_np(env.get_state()), np.stack([tr.worlds[t + 1] for tr in trs]))
        assert np.array_equal(dev_np(obs), np.stack([tr.stables[t + 1] for tr in trs]))
        assert dev_np(rew).tolist() == [int(tr.rewards[t + 1]) for tr in trs]
        assert dev_np(env.last_alive()).tolist() == [int(tr.alives[t + 1]) for tr in trs]
        assert not bool(done.any())
    env.check_actions()


def _random_case(side, n_envs, spawn, smax, seed, steps, BatchedSim, with_actions=True):
    rs = np.random.RandomState(seed)
    size = side * side
    cells = rs.randint(2, size=(n_envs, size)).astype(np.uint8)
    st = rs.randint(-128, 128, size=(n_envs, size)).astype(np.int8)
    env = BatchedSim(n_envs, side, spawnStabilityFactor=spawn, stableStabilityFactor=smax, states=cells)
    env.stable.copy_(torch.from_numpy(st))
    for _ in range(steps):
        acts = rs.randint(size + 1, size=n_envs).astype(np.int32) if with_actions else None
        rew_o, alv_o = oracle.step_batch(cells, st, side, acts, spawn, smax, threads=4)
        obs, rew, _ = env.step(None if acts is None else torch.from_numpy(acts).cuda(), want_alive=True)
        assert np.array_equal(dev_np(env.get_state()), cells), (side, "world")
        assert np.array_equal(dev_np(obs), st), (side, "stable")
        assert np.array_equal(dev_np(rew), rew_o) and np.array_equal(dev_np(env.last_alive()), alv_o.astype(np.int64))
        assert np.array_equal(dev_np(env.reward()), rew_o) and np.array_equal(dev_np(env.alive()), alv_o.astype(np.int64))
    env.check_actions()


@pytest.mark.parametrize("side,n_envs,spawn,smax", [
    (32, 9, -2, 2), (64, 5, -128, 127), (64, 133, -2, 2), (96, 3, 5, 2), (128, 7, -1, 1), (128, 1, 127, -128),
    (160, 2, -2, 2), (192, 2, 0, 0), (224, 1, -3, 100), (256, 3, -2, 2)])
def test_fused_kernel_random_states_vs_oracle(B, side, n_envs, spawn, smax):
    """Arbitrary stability bytes (s > MAX, wrap at 127), random actions incl. the no-op, ragged batch sizes."""
    _random_case(side, n_envs, spawn, smax, seed=side * 7 + n_envs, steps=3, BatchedSim=B)


@pytest.mark.parametrize("side,n_envs", [(1, 4), (2, 3), (3, 5), (5, 2), (7, 33), (10, 64), (31, 3), (33, 2), (40, 9),
                                         (100, 2), (200, 1), (288, 1)])
def test_generic_kernels_random_states_vs_oracle(B, side, n_envs):
    _random_case(side, n_envs, -2, 2, seed=side * 13 + n_envs, steps=3, BatchedSim=B)
    _random_case(side, n_envs, -128, 127, seed=side, steps=2, BatchedSim=B, with_actions=False)


def test_invalid_actions_are_flagged(B):
    env = B(4, 64, spawnStabilityFactor=-2, stableStabilityFactor=2)
    before = dev_np(env.get_state()).copy()
    env.step(torch.tensor([4096, 4097, -1, 4096], dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        env.check_actions()
    env.check_actions()                                  # flag cleared
    cells, st = before.copy(), oracle.initial_stable(before.reshape(-1), -2).reshape(4, -1)
    oracle.step_batch(cells, st, 64, None, -2, 2)        # invalid actions were treated as no-ops
    assert np.array_equal(dev_np(env.get_state()), cells)
    env10 = B(2, 10)
    env10.step(torch.tensor([100, 101], dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        env10.check_actions()


def test_multi_index_toggle_matches_oracle(B):
    rs = np.random.RandomState(5)
    for side in (10, 64):
        size, n = side * side, 7
        cells = rs.randint(2, size=(n, size)).astype(np.uint8)
        st = rs.randint(-128, 128, size=(n, size)).astype(np.int8)
        env = B(n, side, spawnStabilityFactor=-2, stableStabilityFactor=2, states=cells)
        env.stable.copy_(torch.from_numpy(st))
        idx = rs.randint(size, size=(n, 4)).astype(np.int32)
        idx[0] = [3, 3, 3, 9]; idx[1] = [size, 5, size, 5]           # duplicates + no-op padding
        env.toggle(torch.from_numpy(idx).cuda())
        for e in range(n):
            valid = [int(v) for v in idx[e] if v != size]
            oracle.toggle(cells[e], st[e], valid, -2)
        assert np.array_equal(dev_np(env.get_state()), cells) and np.array_equal(dev_np(env.stable), st)
        env.check_actions()


def test_sharding_by_env_index_is_partition_invariant(B):
    """N ranks owning [r*B/G, (r+1)*B/G) produce exactly the rows a single GPU produces."""
    full = B(8, 64, seed=11, spawnStabilityFactor=-2, stableStabilityFactor=2)
    parts = [B.shard(8, 64, r, 4, seed=11, spawnStabilityFactor=-2, stableStabilityFactor=2) for r in range(4)]
    acts = torch.randint(0, 4097, (3, 8), dtype=torch.int32, device="cuda")
    for t in range(3):
        _, rew, _ = full.step(acts[t])
        for r, p in enumerate(parts):
            _, prew, _ = p.step(acts[t, 2 * r:2 * r + 2].contiguous())
            assert torch.equal(prew, rew[2 * r:2 * r + 2])
            assert torch.equal(p.stable, full.stable[2 * r:2 * r + 2])


def test_host_buffer_entry_points(B):
    """cgl_step_state_gpu == the reference's __step_state_gpu contract; step_host == step."""
    from cgl_b200 import native
    lib = native.load()
    for name in ("rand64_plain", "tiny10", "env200_0", "blinker5"):
        tr = TRACES[name]
        w, s = tr.worlds[0].copy(), tr.stables[0].copy()
        for t in range(min(tr.T, 4)):
            a = tr.action(t)
            if a is not None:
                oracle.toggle(w, s, a, tr.spawn)
            native.check(lib.cgl_step_state_gpu(w.ctypes.data, s.ctypes.data, tr.side, tr.spawn, tr.stable_max))
            assert np.array_equal(w, tr.worlds[t + 1]) and np.array_equal(s, tr.stables[t + 1]), (name, t)
    a = B(16, 64, seed=3, spawnStabilityFactor=-2, stableStabilityFactor=2)
    b = B(16, 64, seed=3, spawnStabilityFactor=-2, stableStabilityFactor=2)
    acts_h = torch.empty(16, dtype=torch.int32).pin_memory()
    rew_h = torch.empty(16, dtype=torch.int32).pin_memory()
    obs_h = torch.empty((16, 4096), dtype=torch.int8).pin_memory()
    for t in range(3):
        acts_h.copy_(torch.randint(0, 4097, (16,), dtype=torch.int32))
        a.step_host(acts_h, rew_h, obs_h)
        obs, rew, _ = b.step(acts_h.cuda())
        assert torch.equal(rew.cpu(), rew_h) and torch.equal(obs.cpu(), obs_h)


# ------------------------------------------------------------------------------------------
# life mode (world-only generations of large grids)
# ------------------------------------------------------------------------------------------
def _life_step(lib, native, win, rows, cols, wrap, n_envs=1, want_alive=True):
    out = torch.empty_like(win)
    alive = torch.zeros(n_envs, dtype=torch.int32, device="cuda")
    native.check(lib.cgl_life_step(native.dptr(win), native.dptr(out), n_envs, rows, cols, wrap,
                                   native.dptr(alive) if want_alive else None, native.current_stream()))
    return out, alive


def _pack(lib, native, cells, n_envs, rows, cols):
    W = (cols + 31) // 32
    out = torch.empty(n_envs * rows * W, dtype=torch.int32, device="cuda")
    c = torch.from_numpy(np.ascontiguousarray(cells, np.uint8)).cuda()
    native.check(lib.cgl_pack(native.dptr(c), native.dptr(out), n_envs, rows, cols, native.current_stream()))
    return out


def _unpack(lib, native, w, n_envs, rows, cols):
    out = torch.empty(n_envs * rows * cols, dtype=torch.uint8, device="cuda")
    native.check(lib.cgl_unpack(native.dptr(w), native.dptr(out), n_envs, rows, cols, native.current_stream()))
    return out.cpu().numpy()


@pytest.mark.parametrize("rows,cols,n_envs", [(50, 2048, 1), (131, 4096, 1), (64, 4096 + 128 * 5, 2), (300, 8192, 1),
                                              (17, 100, 3), (9, 2176, 1)])
@pytest.mark.parametrize("wrap", [1, 0])
def test_life_step_vs_oracle(cgl, rows, cols, n_envs, wrap):
    from cgl_b200 import native
    lib = native.load()
    rs = np.random.RandomState(rows + cols)
    cells = rs.randint(2, size=(n_envs, rows, cols)).astype(np.uint8)
    w = _pack(lib, native, cells, n_envs, rows, cols)
    for g in range(3):
        w, alive = _life_step(lib, native, w, rows, cols, wrap, n_envs)
        for e in range(n_envs):
            if wrap:
                cells[e] = oracle.life(cells[e], 1, threads=4)
            else:       # dead rows outside, torus columns == torus on a grid padded with 2 dead rows, re-killed
                padded = np.zeros((rows + 2, cols), np.uint8)
                padded[1:-1] = cells[e]
                cells[e] = oracle.life(padded, 1, threads=4)[1:-1]
        got = _unpack(lib, native, w, n_envs, rows, cols).reshape(n_envs, rows, cols)
        assert np.array_equal(got, cells), (rows, cols, wrap, g)
        assert (alive.cpu().numpy().astype(np.int64) & 0xFFFFFFFF).tolist() == cells.reshape(n_envs, -1).sum(1).tolist()


# ------------------------------------------------------------------------------------------
# temporal blocking: k generations per launch (cgl_life_run)
# ------------------------------------------------------------------------------------------
def _life_run(lib, native, a, rows, cols, wrap, gens, k):
    b = torch.empty_like(a)
    res = native.ctypes.c_int(-1)
    native.check(lib.cgl_life_run(native.dptr(a), native.dptr(b), rows, cols, wrap, gens, k,
                                  native.ctypes.byref(res), native.current_stream()))
    return a if res.value == 1 else b


@pytest.mark.parametrize("rows,cols,gens,k", [(200, 1024, 8, 8), (97, 2048, 13, 4), (64, 960, 5, 2), (300, 4096, 32, 16),
                                              (128, 1920, 7, 3), (50, 1024, 12, 12), (40, 992, 6, 6), (33, 3104, 9, 1)])
def test_temporal_blocking_torus_vs_oracle(cgl, rows, cols, gens, k):
    from cgl_b200 import native
    lib = native.load()
    cells = np.random.RandomState(rows * 7 + cols + k).randint(2, size=(rows, cols)).astype(np.uint8)
    a = _pack(lib, native, cells, 1, rows, cols)
    out = _life_run(lib, native, a, rows, cols, 1, gens, k)
    got = _unpack(lib, native, out, 1, rows, cols).reshape(rows, cols)
    assert np.array_equal(got, oracle.life(cells, gens, threads=4))


@pytest.mark.parametrize("rows,cols,k", [(120, 1024, 8), (90, 2048, 4), (200, 960, 16)])
def test_temporal_blocking_open_band_interior(cgl, rows, cols, k):
    """wrap_rows=0, one k-block: every row at least k rows from an open edge is exact (ghost-zone contract)."""
    from cgl_b200 import native
    lib = native.load()
    cells = np.random.RandomState(rows + k).randint(2, size=(rows, cols)).astype(np.uint8)
    a = _pack(lib, native, cells, 1, rows, cols)
    out = _life_run(lib, native, a, rows, cols, 0, k, k)
    got = _unpack(lib, native, out, 1, rows, cols).reshape(rows, cols)
    padded = np.zeros((rows + 2 * k + 2, cols), np.uint8)
    padded[k + 1:k + 1 + rows] = cells
    want = oracle.life(padded, k, threads=4)[k + 1:k + 1 + rows]
    assert np.array_equal(got[k:rows - k], want[k:rows - k])


# ------------------------------------------------------------------------------------------
# opt-in kernel variants stay parity-green (selected by environment knobs, so run in a subprocess)
# ------------------------------------------------------------------------------------------
_VARIANT_SCRIPT = r"""
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
from cgl_b200.batched import BatchedSim
from oracle import oracle
for side, n in ((128, 9), (64, 37), (32, 70), (10, 40), (33, 9), (50, 21), (100, 6), (131, 3), (200, 4), (1, 5), (3, 7)):
    size = side * side
    rs = np.random.RandomState(side)
    cells = rs.randint(2, size=(n, size)).astype(np.uint8)
    st = rs.randint(-128, 128, size=(n, size)).astype(np.int8)
    env = BatchedSim(n, side, spawnStabilityFactor=-2, stableStabilityFactor=2, states=cells)
    env.stable.copy_(torch.from_numpy(st))
    for _ in range(3):
        acts = rs.randint(size + 1, size=n).astype(np.int32)
        rew_o, alv_o = oracle.step_batch(cells, st, side, acts, -2, 2, threads=4)
        obs, rew, _ = env.step(torch.from_numpy(acts).cuda(), want_alive=True)
        assert np.array_equal(env.get_state().cpu().numpy(), cells)
        assert np.array_equal(obs.cpu().numpy(), st)
        assert np.array_equal(rew.cpu().numpy(), rew_o)
        assert np.array_equal(env.last_alive().cpu().numpy(), alv_o.astype(np.int64))
print("variant ok")
"""


@pytest.mark.parametrize("knobs", [{"CGL_ENV_PDL": "0"}, {"CGL_ENV_BYTES": "0"}, {"CGL_ENV_BYTES": "2"}])
def test_env_kernel_variants_vs_oracle(cgl, knobs):
    """The non-PDL launch path and -- on sides the fused kernel does not take -- the one-launch byte-plane kernel
    against the three generic kernels it replaced."""
    import subprocess
    import sys
    from conftest import PKG
    env = dict(os.environ, **knobs)
    r = subprocess.run([sys.executable, "-c", _VARIANT_SCRIPT, ROOT, PKG], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "variant ok" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


def test_facade_reference_attributes(cgl):
    """Attribute names scripts of the reference touch directly (world, stable, initState, initStable, ...)."""
    tr = TRACES["tiny10"]
    env = cgl.sim(state=tr.worlds[0].reshape(10, 10), gpu=True, spawnStabilityFactor=tr.spawn,
                  stableStabilityFactor=tr.stable_max)
    assert np.array_equal(env.world, tr.worlds[0]) and np.array_equal(env.stable, tr.stables[0])
    assert np.array_equal(env.initState, tr.worlds[0]) and np.array_equal(env.initStable, tr.stables[0])
    assert (env.size, env.side, env.count, env.gpu) == (100, 10, 0, True)
    env.toggle_state(np.int32(tr.action(0)))
    assert env.reward() == tr.rewards_after_toggle[0]          # deferred toggle is visible to reward()
    env.step()
    assert np.array_equal(env.world, tr.worlds[1]) and np.array_equal(env.stable, tr.stables[1])
    assert np.array_equal(env.initState, tr.worlds[0])         # reset source untouched
    env.toggle_state(np.int32(tr.action(1)))
    env.toggle_state(np.int32(tr.action(1)))                   # two deferred toggles of one cell cancel in the world ...
    w = env.get_state(vector=True)
    assert np.array_equal(w, tr.worlds[1])
    assert env.get_stable(vector=True)[tr.action(1)] == tr.spawn or tr.action(1) == 100   # ... but stable = spawn


def test_async_host_step_two_groups_equal_sync_steps(cgl):
    """cgl_env_step_host_async + cgl_stream_wait: two env groups on two streams, double-buffered, give the same
    observations and rewards as synchronous host steps of the same envs."""
    from cgl_b200.batched import BatchedSim
    side, n = 64, 96
    size = side * side
    rs = np.random.RandomState(4)
    sync_env = BatchedSim(2 * n, side, seed=9, spawnStabilityFactor=-2, stableStabilityFactor=2)
    groups = [BatchedSim(n, side, seed=9, first_env=g * n, spawnStabilityFactor=-2, stableStabilityFactor=2) for g in range(2)]
    streams = [torch.cuda.Stream() for _ in range(2)]
    acts_all = torch.empty(2 * n, dtype=torch.int32).pin_memory()
    rew_all = torch.empty(2 * n, dtype=torch.int32).pin_memory()
    acts_g = [torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(2)]
    rew_g = [torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(2)]
    torch.cuda.synchronize()
    for t in range(6):
        a = rs.randint(0, size + 1, size=2 * n).astype(np.int32)
        acts_all.numpy()[:] = a
        sync_env.step_host(acts_all, rew_all)
        for g in range(2):
            with torch.cuda.stream(streams[g]):
                groups[g].wait_host()
                acts_g[g].numpy()[:] = a[g * n:(g + 1) * n]
                groups[g].step_host(acts_g[g], rew_g[g], sync=False)
        for g in range(2):
            with torch.cuda.stream(streams[g]):
                groups[g].wait_host()
            assert np.array_equal(rew_g[g].numpy(), rew_all.numpy()[g * n:(g + 1) * n]), (t, g)
            assert torch.equal(groups[g].stable, sync_env.stable[g * n:(g + 1) * n])


@pytest.mark.parametrize("kw", [dict(side=64), dict(side=10), dict(side=32, dead_rule="decay", empty=-1, empty_min=-5, masked_toggle=True)])
def test_checkpoint_resume_continues_bit_for_bit(cgl, tmp_path, kw):
    from cgl_b200.batched import BatchedSim
    side = kw.pop("side")
    n, size = 40, side * side
    env = BatchedSim(n, side, seed=6, spawnStabilityFactor=-2, stableStabilityFactor=2, rng="device", max_steps=6, **kw)
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    acts = [torch.randint(0, size + 1, (n,), dtype=torch.int32, device="cuda", generator=g) for _ in range(8)]
    for a in acts[:3]:
        env.step(a)
    path = str(tmp_path / "batch.npz")
    env.save_checkpoint(path)
    twin = BatchedSim.load_checkpoint(path)
    assert twin.count == env.count == 3 and twin.dead_rule == env.dead_rule and twin.masked_toggle == env.masked_toggle
    assert torch.equal(twin.world, env.world) and torch.equal(twin.stable, env.stable)
    assert twin.max_steps == 6 and twin.rng == "device"                     # (format v2: the `done` horizon travels too)
    for a in acts[3:]:
        oa, ra, da = env.step(a)
        ob, rb, db = twin.step(a)
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(env.world, twin.world)
        assert torch.equal(da, db) and bool(da.all()) == (env.count >= 6)
    env.reset(); twin.reset()
    assert torch.equal(env.world, twin.world) and torch.equal(env.stable, twin.stable)
    with pytest.raises(ValueError):
        np.savez(str(tmp_path / "bad.npz"), format=np.array("something else"))
        BatchedSim.load_checkpoint(str(tmp_path / "bad.npz"))


@pytest.mark.parametrize("rows,cols,n_envs", [(128, 128, 7), (64, 64, 33), (3, 4096, 2), (37, 160, 5), (50, 50, 3), (9, 33, 4)])
def test_pack_unpack_and_initial_stability_at_the_api_boundary(cgl, rows, cols, n_envs):
    """cgl_pack / cgl_unpack / cgl_init_stable(_rule): the whole-word fast kernels (cols % 32 == 0, 16-byte aligned
    buffers), the same data through a misaligned view (generic kernels), and ragged widths -- against numpy.
    Cells arrive as arbitrary bytes: nonzero = alive (CGL/CGL.py:94,107,111-112; fork: CGL_action+/CGL.py:122-126)."""
    import torch
    from cgl_b200 import native
    lib = native.load()
    rs = np.random.RandomState(rows * 1000 + cols)
    cells = (rs.randint(0, 4, size=(n_envs, rows * cols)) * rs.randint(1, 64, size=(n_envs, rows * cols))).astype(np.uint8)
    alive = (cells != 0).astype(np.uint8)
    W = (cols + 31) // 32
    st = native.current_stream()
    for misalign in (0, 1):
        raw = torch.zeros(cells.size + 16, dtype=torch.uint8, device="cuda")
        c_d = raw[misalign:misalign + cells.size]
        c_d.copy_(torch.from_numpy(cells.reshape(-1)))
        world = torch.zeros(n_envs * rows * W, dtype=torch.int32, device="cuda")
        native.check(lib.cgl_pack(native.dptr(c_d), native.dptr(world), n_envs, rows, cols, st))
        out_raw = torch.full((cells.size + 16,), 7, dtype=torch.uint8, device="cuda")
        out = out_raw[misalign:misalign + cells.size]
        native.check(lib.cgl_unpack(native.dptr(world), native.dptr(out), n_envs, rows, cols, st))
        assert np.array_equal(out.cpu().numpy().reshape(n_envs, -1), alive), (rows, cols, misalign)
        assert int(out_raw[misalign + cells.size:].min()) == 7 and (misalign == 0 or int(out_raw[0]) == 7)
        if rows == cols:
            for spawn, empty in ((-2, 0), (0, -3), (5, -1), (-128, 127)):
                s_raw = torch.zeros(cells.size + 16, dtype=torch.int8, device="cuda")
                s_d = s_raw[misalign:misalign + cells.size]
                native.check(lib.cgl_init_stable_rule(native.dptr(world), native.dptr(s_d), n_envs, rows, spawn, empty, st))
                want = np.where(alive == 1, np.int8(spawn), np.int8(0)).astype(np.int8)
                want[want == 0] = np.int8(empty)
                assert np.array_equal(s_d.cpu().numpy().reshape(n_envs, -1), want), (rows, spawn, empty, misalign)
                native.check(lib.cgl_init_stable(native.dptr(world), native.dptr(s_d), n_envs, rows, spawn, st))
                assert np.array_equal(s_d.cpu().numpy().reshape(n_envs, -1),
                                      np.where(alive == 1, np.int8(spawn), np.int8(0))), (rows, spawn, misalign)
