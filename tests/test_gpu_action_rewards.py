"""GPU suite: every action's next-step reward and the greedy action (cgl_env_action_rewards).

  * the map equals the host restatement (tests/oracle_lookahead.py) env by env on every fused side and on generic
    sides 1 to 300, all three dead-cell rules, masked and unmasked toggles, batches with partial CTAs, dense and sparse
    soups, an empty and a full world, random int8 planes;
  * map[e, a[e]] equals the reward step(a) returns on an identical env, and column `size` equals step(None)'s;
  * greedy_actions equals map.argmax(1) / map.max(1) exactly, ties included; the planes and `count` are untouched;
  * a map past 2^32 bytes is right in its last rows (64-bit offsets);
  * the torch extension equals the ctypes path; both facades' action_rewards() match the restatement after a deferred
    toggle, after lazy steps and while the resident step server is serving.
"""
import importlib.util
import os

import numpy as np
import pytest

from conftest import PKG
from oracle import oracle
import oracle_lookahead as look

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

RULE_ID = {"zero": oracle.DEAD_ZERO, "decay": oracle.DEAD_DECAY, "sat": oracle.DEAD_SAT}
FUSED = [32, 64, 96, 128, 160, 192, 224, 256]
GENERIC = [1, 2, 3, 10, 17, 33, 100, 200, 257, 300]
VARIANTS = [("zero", False, -1, 1, 0, -128), ("zero", True, -2, 2, 0, -128), ("decay", True, -2, 3, -1, -6),
            ("sat", False, 100, -100, 120, 7), ("decay", False, -128, 127, 0, -128)]


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200 import native
    native.load()
    return torch.device("cuda", 0)


def boards(rs, B, side):
    """B boards: a dense soup, a sparse soup, an empty world, a full world, then soups of random density."""
    size = side * side
    dens = [0.5, 0.08, 0.0, 1.0] + list(rs.uniform(0.05, 0.6, size=max(0, B - 4)))
    return np.stack([(rs.rand(size) < d).astype(np.uint8) for d in dens[:B]])


def make_env(cuda, B, side, rule, masked, spawn, smax, empty, emin, seed, random_plane=True):
    from cgl_b200.batched import BatchedSim
    rs = np.random.RandomState(seed)
    cells = boards(rs, B, side)
    env = BatchedSim(B, side, spawnStabilityFactor=spawn, stableStabilityFactor=smax, device=cuda, states=cells,
                     dead_rule=rule, empty=empty, empty_min=emin, masked_toggle=masked)
    if random_plane:
        env.stable.copy_(torch.from_numpy(rs.randint(-128, 128, size=(B, side * side)).astype(np.int8)))
    return env


def host_state(env):
    return env.get_state().cpu().numpy(), env.stable.cpu().numpy()


def check_env(env, rule, masked, spawn, smax, empty, emin):
    worlds, stables = host_state(env)
    w_before, s_before, count = env._wa.clone(), env.stable.clone(), env.count
    m = env.action_rewards()
    act, rew = env.greedy_actions()
    torch.cuda.synchronize()
    want = look.batch(worlds, stables, env.side, spawn, smax, RULE_ID[rule], empty, emin, masked)
    got = m.cpu().numpy()
    for e in range(env.n_envs):
        assert np.array_equal(got[e], want[e]), (env.side, rule, masked, e, np.nonzero(got[e] != want[e])[0][:8])
    assert np.array_equal(act.cpu().numpy(), want.argmax(1)) and np.array_equal(rew.cpu().numpy(), want.max(1))
    assert torch.equal(env._wa, w_before) and torch.equal(env.stable, s_before) and env.count == count


@pytest.mark.parametrize("side", FUSED + GENERIC)
@pytest.mark.parametrize("variant", VARIANTS, ids=lambda v: f"{v[0]}-{'masked' if v[1] else 'plain'}-{v[2]}")
def test_map_equals_restatement(cuda, side, variant):
    rule, masked, spawn, smax, empty, emin = variant
    B = 6 if side <= 64 else 5                              # partial CTAs where several envs share one
    env = make_env(cuda, B, side, rule, masked, spawn, smax, empty, emin, seed=side)
    check_env(env, rule, masked, spawn, smax, empty, emin)
    # the env's own initial planes (stability = SPAWN / EMPTY, no random plane)
    env = make_env(cuda, B, side, rule, masked, spawn, smax, empty, emin, seed=side + 1, random_plane=False)
    check_env(env, rule, masked, spawn, smax, empty, emin)


@pytest.mark.parametrize("B", [1, 3, 4, 5, 9, 150])
@pytest.mark.parametrize("side", [32, 64, 128])
def test_batch_sizes(cuda, side, B):
    env = make_env(cuda, B, side, "zero", False, -1, 1, 0, -128, seed=B)
    check_env(env, "zero", False, -1, 1, 0, -128)


@pytest.mark.parametrize("side", [128, 256, 100])
@pytest.mark.parametrize("rule,masked", [("zero", False), ("decay", True), ("sat", True)])
def test_map_against_gpu_steps(cuda, side, rule, masked):
    """map[e, a[e]] is what step(a) returns on an identical env; column size is what step(None) returns."""
    from cgl_b200.batched import BatchedSim
    B = 48
    env = make_env(cuda, B, side, rule, masked, -2, 3, -1, -7, seed=side + 5)
    m = env.action_rewards().cpu().numpy()
    rs = np.random.RandomState(side)
    for trial in range(4):
        acts = rs.randint(side * side + 1, size=B).astype(np.int32)
        if trial == 0:
            acts[:] = side * side
        twin = BatchedSim(B, side, spawnStabilityFactor=-2, stableStabilityFactor=3, device=cuda,
                          states=env.get_state().cpu().numpy(), dead_rule=rule, empty=-1, empty_min=-7, masked_toggle=masked)
        twin.stable.copy_(env.stable)
        _, rew, _ = twin.step(torch.from_numpy(acts).to(cuda))
        assert np.array_equal(rew.cpu().numpy(), m[np.arange(B), acts]), (side, rule, trial)


def test_greedy_ties_and_caller_buffers(cuda):
    """Boards whose best reward is shared by many actions: the smallest index wins, like torch.argmax."""
    from cgl_b200.batched import BatchedSim
    side, B = 64, 5
    cells = np.zeros((B, side * side), np.uint8)
    for e in range(1, B):                                   # blocks (still lifes) at different places
        r, c = 5 * e, 7 * e
        for dy, dx in ((0, 0), (0, 1), (1, 0), (1, 1)):
            cells[e, (r + dy) * side + c + dx] = 1
    env = BatchedSim(B, side, spawnStabilityFactor=-1, stableStabilityFactor=1, device=cuda, states=cells)
    m = env.action_rewards()
    assert all(int((row == row.max()).sum()) > 1 for row in m.cpu().numpy())
    out = torch.full((B,), -5, dtype=torch.int32, device=cuda)
    rout = torch.full((B,), -5, dtype=torch.int32, device=cuda)
    a, r = env.greedy_actions(out=out, reward_out=rout)
    assert a is out and r is rout
    assert torch.equal(a.long(), m.argmax(1)) and torch.equal(r, m.max(1).values)
    mo = torch.empty((B, side * side + 1), dtype=torch.int32, device=cuda)
    assert env.action_rewards(out=mo) is mo and torch.equal(mo, m)
    with pytest.raises(TypeError):
        env.action_rewards(out=torch.empty((B, side * side), dtype=torch.int32, device=cuda))
    with pytest.raises(TypeError):
        env.greedy_actions(out=torch.empty(B, dtype=torch.int32))


def test_map_past_4_gib(cuda):
    """65536 envs x 128^2: the map is 4.29 GB, so its last rows need 64-bit offsets."""
    from cgl_b200.batched import BatchedSim
    B, side = 65536, 128
    env = BatchedSim(B, side, spawnStabilityFactor=-2, stableStabilityFactor=2, device=cuda, rng="device", seed=9)
    m = torch.full((B, side * side + 1), 7, dtype=torch.int32, device=cuda)
    env.action_rewards(out=m)
    a, r = env.greedy_actions()
    rows = [0, 1, 32767, B - 3, B - 2, B - 1]
    cells = env.get_state()[rows].cpu().numpy()
    st = env.stable[rows].cpu().numpy()
    want = look.batch(cells, st, side, -2, 2)
    got = m[rows].cpu().numpy()
    assert np.array_equal(got, want)
    assert np.array_equal(a[rows].cpu().numpy(), want.argmax(1)) and np.array_equal(r[rows].cpu().numpy(), want.max(1))
    del m


@pytest.mark.parametrize("side", [64, 100])
def test_torch_extension_equals_ctypes(cuda, side):
    from cgl_b200 import native
    env = make_env(cuda, 7, side, "decay", True, -2, 3, -1, -6, seed=3)
    m = env.action_rewards()
    a, r = env.greedy_actions()
    ext = native.ext()
    m2 = torch.empty_like(m)
    a2, r2 = torch.empty_like(a), torch.empty_like(r)
    ext.env_action_rewards(env._wa, env.stable, side, spawn=-2, stable_max=3, dead_rule=1, empty=-1, empty_min=-6,
                           masked_toggle=True, rewards_out=m2)
    ext.env_action_rewards(env._wa, env.stable, side, spawn=-2, stable_max=3, dead_rule=1, empty=-1, empty_min=-6,
                           masked_toggle=True, best_action_out=a2, best_reward_out=r2)
    assert torch.equal(m, m2) and torch.equal(a, a2) and torch.equal(r, r2)
    with pytest.raises(RuntimeError):
        ext.env_action_rewards(env._wa, env.stable, side)                 # no output
    with pytest.raises(RuntimeError):
        ext.env_action_rewards(env._wa, env.stable, side, rewards_out=m2[:, 1:].contiguous())


@pytest.fixture(scope="module")
def CGL(cuda):
    import CGL as mod
    return mod


@pytest.fixture(scope="module")
def fork(cuda):
    spec = importlib.util.spec_from_file_location("cgl_fork_facade_look", os.path.join(PKG, "CGL_action+", "CGL.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _facade_check(env, ref, rule, masked, empty, emin):
    got = env.action_rewards()
    assert got.dtype == np.int32 and got.shape == (ref.size + 1,)
    want = look.action_rewards(ref.world, ref.stable, ref.side, ref.spawn, ref.smax, rule, empty, emin, masked)
    assert np.array_equal(got, want)


class _Ref:
    """The oracle env the facade is compared with (toggle / step with the same rule)."""

    def __init__(self, world, stable, side, spawn, smax, rule, empty, emin, masked):
        self.world, self.stable, self.side, self.size = world.copy(), stable.copy(), side, side * side
        self.spawn, self.smax, self.rule, self.empty, self.emin, self.masked = spawn, smax, rule, empty, emin, masked

    def toggle(self, a):
        (oracle.toggle_masked if self.masked else oracle.toggle)(self.world, self.stable, a, self.spawn)

    def step(self):
        oracle.step_rule(self.world, self.stable, self.side, self.spawn, self.smax, self.rule, self.empty, self.emin)


@pytest.mark.parametrize("side", [2, 10, 64, 128, 300])
def test_base_facade(CGL, side):
    env = CGL.sim(side=side, seed=4, gpu=True, spawnStabilityFactor=-2, stableStabilityFactor=2)
    ref = _Ref(env.get_state(vector=True), env.get_stable(vector=True), side, -2, 2, 0, 0, -128, False)
    _facade_check(env, ref, 0, False, 0, -128)
    rs = np.random.RandomState(side)
    a = int(rs.randint(side * side))
    env.toggle_state(a); ref.toggle(a)                     # deferred toggle
    _facade_check(env, ref, 0, False, 0, -128)
    for _ in range(3):                                     # lazy plain steps
        env.step(); ref.step()
    _facade_check(env, ref, 0, False, 0, -128)
    for _ in range(5):                                     # the DQN loop (served steps where the server takes the side)
        a = int(rs.randint(side * side + 1))
        env.toggle_state(a); env.step()
        if a < side * side:
            ref.toggle(a)
        ref.step()
        obs = env.get_stable(vector=True, shallow=True)
        assert int(env.reward()) == int(oracle.reward(ref.stable))
    served = env._serving
    _facade_check(env, ref, 0, False, 0, -128)
    assert not env._serving
    if side <= 256:
        assert served
    assert np.array_equal(obs, ref.stable)


@pytest.mark.parametrize("side", [10, 64])
@pytest.mark.parametrize("rule", ["decay", "sat"])
def test_fork_facade(fork, side, rule):
    env = fork.sim(side=side, seed=2, gpu=True, spawnStabilityFactor=-2, stableStabilityFactor=3, empty=-1,
                   empty_min=-6, dead_rule=rule)
    ref = _Ref(env.get_state(vector=True), env.get_stable(vector=True), side, -2, 3, RULE_ID[rule], -1, -6, True)
    _facade_check(env, ref, RULE_ID[rule], True, -1, -6)
    rs = np.random.RandomState(side)
    for _ in range(4):
        a = int(rs.randint(side * side))
        env.toggle_state(a); env.step()
        ref.toggle(a); ref.step()
        env.get_stable(vector=True, shallow=True)
    a = int(rs.randint(side * side))
    env.toggle_state(a); ref.toggle(a)
    _facade_check(env, ref, RULE_ID[rule], True, -1, -6)
    assert env.get_count() == 4
