"""GPU suite: the single-env paths that the reference's own training loop takes (CGL/main.py:64-72), against the oracle.

`CGL.sim` -> toggle_state -> step -> get_stable -> reward runs on kernels of its own, each of which restates the
generation and the stability rule:
  * `sim1_step_kernel` (cgl_sim_step / cgl_sim_step_ex, sides <= 448) and the resident `sim1_serve_kernel`
    (cgl_sim_serve, sides <= 256), both with a side-dependent thread layout (four cells per thread, ceil(side / 4)
    threads per row, 1024 / that rows per pass, a byte path where side % 4 != 0);
  * the facades' four regimes: served (1-256), one-launch steps plus deferred on-chip runs (257-274), one-launch
    steps only (275-448), the batched kernels (449 and above);
  * the host-driven rollout (cgl_rollout_*, zero-copy actions or an H2D copy node; rewards direct or through a D2H
    copy node) and the host-buffer entry points (cgl_env_step_host / _async, cgl_step_state_gpu).
Everything is compared bit for bit with the C oracle through tests/oracle_facade.py, at every side where a layout
changes and at the parameter corners of oracle_facade.CORNERS on arbitrary int8 stability planes.
"""
import ctypes
import importlib.util
import os
import time

import numpy as np
import pytest

from conftest import PKG
from oracle import oracle
from oracle_facade import BASE_CORNERS, CORNERS, FORK_CORNERS, OracleEnv, corner_plane

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

LAYOUT_SIDES = [1, 2, 3, 4, 5, 7, 31, 32, 33, 63, 64, 65, 100, 127, 128, 129, 255, 256, 257, 447, 448]
RULE_NAME = {oracle.DEAD_DECAY: "decay", oracle.DEAD_SAT: "sat"}
LINGER_US = 100000                  # the longest a served launch waits for a command before it leaves by itself
WAIT_S = 10.0                       # bound of every host-side wait for the device


@pytest.fixture(scope="module")
def native():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200 import native as mod
    mod.load()
    return mod


@pytest.fixture(scope="module")
def CGL(native):
    import CGL as mod
    return mod


@pytest.fixture(scope="module")
def fork(native):
    spec = importlib.util.spec_from_file_location("cgl_fork_facade_single_env", os.path.join(PKG, "CGL_action+", "CGL.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def edge_actions(rs, side):
    """The no-op, cell 0, the last cell, the last cell of a row, a cell of a row's partial last group of four (if the
    side has one) and one random action."""
    size = side * side
    acts = [0, size - 1, int(rs.randint(side)) * side + side - 1]
    if side % 4:
        acts.append(int(rs.randint(side)) * side + side - 1 - int(rs.randint(side % 4)))
    return acts + [size, int(rs.randint(size + 1))]


def oracle_step(cells, st, side, corner, a):
    spawn, smax, rule, empty, emin, masked = corner
    if a < side * side:
        (oracle.toggle_masked if masked else oracle.toggle)(cells, st, a, spawn)
    oracle.step_rule(cells, st, side, spawn, smax, rule, empty, emin)


def wait_until(cond, what):
    t0 = time.perf_counter()
    while not cond():
        if time.perf_counter() - t0 > WAIT_S:
            raise AssertionError(f"timed out: {what}")


class SingleEnv:
    """One env's device planes, pinned observation mirror and pinned result block, and the cgl_sim_step_args_t over
    them.  The world sits in world_a if the flip counter is even, else in world_b."""

    def __init__(self, native, side, corner, cells, st, flip=0, mirror=True):
        self.native, self.lib = native, native.load()
        self.side, self.size = side, side * side
        W = (side + 31) // 32
        self.planes = [torch.zeros(side * W, dtype=torch.int32, device="cuda") for _ in range(2)]
        self.stable = torch.from_numpy(st.copy()).cuda()
        self.mirror = torch.zeros(self.size, dtype=torch.int8).pin_memory() if mirror else None
        self.res_t = torch.zeros(8, dtype=torch.int32).pin_memory()
        self.res = self.res_t.numpy()
        self.flip = ctypes.c_uint32(flip)
        a = native.SimStepArgs()
        a.world_a, a.world_b, a.stable = self.planes[0].data_ptr(), self.planes[1].data_ptr(), self.stable.data_ptr()
        a.side = side
        a.spawn, a.stable_max, a.dead_rule, a.empty, a.empty_min, masked = corner
        a.masked_toggle = int(masked)
        a.obs_mirror = None if self.mirror is None else self.mirror.data_ptr()
        a.result = self.res_t.data_ptr()
        a.flip_planes = ctypes.pointer(self.flip)
        self.args = a
        self.put_world(cells)

    def put_world(self, cells):
        """Pack `cells` into the plane that holds the world; fill the other plane with random bits."""
        cur = self.flip.value & 1
        c_d = torch.from_numpy(np.ascontiguousarray(cells)).cuda()
        self.native.check(self.lib.cgl_pack(self.native.dptr(c_d), self.native.dptr(self.planes[cur]), 1, self.side,
                                            self.side, self.native.current_stream()), "cgl_pack")
        self.planes[cur ^ 1].random_(-2 ** 31, 2 ** 31 - 1)
        torch.cuda.synchronize()

    def world(self, plane=None):
        p = self.planes[self.flip.value & 1 if plane is None else plane]
        out = torch.empty(self.size, dtype=torch.uint8, device="cuda")
        self.native.check(self.lib.cgl_unpack(self.native.dptr(p), self.native.dptr(out), 1, self.side, self.side,
                                              self.native.current_stream()), "cgl_unpack")
        return out.cpu().numpy()


# ------------------------------------------------------------------------------------------------------------------
# 1. cgl_sim_step_ex: every side up to the limit, and every corner on the sides where the layout changes
# ------------------------------------------------------------------------------------------------------------------
def sim_step_case(native, side, corner, rs, actions, flip, seq0):
    cells = rs.randint(2, size=side * side).astype(np.uint8)
    st = corner_plane(rs, side * side, corner)
    env = SingleEnv(native, side, corner, cells, st, flip=flip)
    lib = env.lib
    for t, a in enumerate(actions):
        env.mirror.numpy()[:] = ~st                          # poison: every byte the step must rewrite differs
        env.res[:4] = (-7, -7, -7, -7)
        seq = seq0 + t
        native.check(lib.cgl_sim_step_ex(ctypes.byref(env.args), a, seq, native.current_stream()), "cgl_sim_step_ex")
        torch.cuda.synchronize()
        oracle_step(cells, st, side, corner, a)
        what = (side, corner, t, a)
        assert env.flip.value == flip + t + 1, what
        assert np.array_equal(env.world(), cells), what
        assert np.array_equal(env.stable.cpu().numpy(), st), what
        assert np.array_equal(env.mirror.numpy(), st), what
        assert (int(env.res[0]), int(env.res[1]), int(env.res[2]) & 0xFFFFFFFF) == \
            (int(oracle.reward(st)), int(oracle.alive(cells)), seq), what


@pytest.mark.parametrize("side", range(1, 449))
def test_sim_step_every_side(native, side):
    """Every side 1..448 at the corner side % 23: each corner meets each side % 4 class and both one and several row
    passes (the boundary is 64 -> 65); odd sides start with the world in world_b."""
    rs = np.random.RandomState(side)
    corner = CORNERS[side % len(CORNERS)]
    sim_step_case(native, side, corner, rs, edge_actions(rs, side), side & 1, 1 + 7 * side)


@pytest.mark.parametrize("side", LAYOUT_SIDES)
def test_sim_step_every_corner_on_layout_sides(native, side):
    rs = np.random.RandomState(1000 + side)
    for ci, corner in enumerate(CORNERS):
        acts = edge_actions(rs, side)
        acts = [acts[(ci + k) % len(acts)] for k in range(3)]
        sim_step_case(native, side, corner, rs, acts, ci & 1, 0x7ffffff0 + 3 * ci)


# ------------------------------------------------------------------------------------------------------------------
# 2. cgl_sim_serve through the C-ABI mailbox
# ------------------------------------------------------------------------------------------------------------------
def serve_session(native, env, corner, cells, st, actions, last_seq, launch_id, stream):
    """Launch the server on `stream` (own, non-blocking, never synchronised while a command is outstanding), serve
    `actions` checking every answer, then QUIT.  A failing check still ends the launch: QUIT, or at worst the linger.
    Returns the last sequence number used."""
    lib, side = env.lib, env.side
    cmd_t = torch.zeros(2, dtype=torch.int64).pin_memory()
    cmd = cmd_t.numpy().view(np.uint64)
    cmd[0] = last_seq << 32                                  # the command already served: not new
    env.res[:] = 0
    env.res[4] = launch_id + 1000
    res = env.res
    torch.cuda.synchronize()                                 # the planes are in place before the server reads them
    native.check(lib.cgl_sim_serve(ctypes.byref(env.args), cmd_t.data_ptr(), last_seq, launch_id, LINGER_US,
                                   stream.cuda_stream), "cgl_sim_serve")
    seq, left = last_seq, False
    try:
        for a in actions:
            if env.mirror is not None:
                env.mirror.numpy()[:] = ~st                  # the server is idle between commands: safe to poison
            seq += 1
            cmd[0] = (seq << 32) | a
            wait_until(lambda: int(res[2]) == seq or int(res[4]) == launch_id, f"side {side}: no answer to {seq}")
            assert int(res[2]) == seq, f"side {side}: the server left before it answered command {seq}"
            oracle_step(cells, st, side, corner, a)
            what = (side, corner, seq, a)
            assert (int(res[0]), int(res[1])) == (int(oracle.reward(st)), int(oracle.alive(cells))), what
            if env.mirror is not None:
                assert np.array_equal(env.mirror.numpy(), st), what
        seq += 1
        cmd[0] = (seq << 32) | native.SIM_QUIT
        wait_until(lambda: int(res[4]) == launch_id, f"side {side}: the server did not leave")
        left = True
    finally:
        if not left:
            seq += 1
            cmd[0] = (seq << 32) | native.SIM_QUIT
            t0 = time.perf_counter()
            while int(res[4]) != launch_id and time.perf_counter() - t0 < WAIT_S:
                pass
    stream.synchronize()                                     # it has left: nothing is outstanding
    return seq


def serve_case(native, side, corner, rs, stream, mirror=True):
    size = side * side
    cells = rs.randint(2, size=size).astype(np.uint8)
    st = corner_plane(rs, size, corner)
    env = SingleEnv(native, side, corner, cells, st, flip=0, mirror=mirror)
    seq = serve_session(native, env, corner, cells, st, edge_actions(rs, side), 5 * side, 1, stream)
    assert np.array_equal(env.world(0), cells) and np.array_equal(env.stable.cpu().numpy(), st), (side, corner)
    # relaunch with the state in world_b (an odd flip counter); world_a is garbage and must stay untouched
    env.flip.value = 1
    env.put_world(cells)
    garbage = env.planes[0].clone()
    serve_session(native, env, corner, cells, st, [int(rs.randint(size + 1)), size, int(rs.randint(size))], seq, 2,
                  stream)
    assert env.flip.value == 1                               # cgl_sim_serve does not advance the counter
    assert np.array_equal(env.world(1), cells) and np.array_equal(env.stable.cpu().numpy(), st), (side, corner)
    assert torch.equal(env.planes[0], garbage)


@pytest.fixture(scope="module")
def serve_stream(native):
    return torch.cuda.Stream()                               # torch's pool streams are non-blocking


@pytest.mark.parametrize("side", range(1, 257))
def test_serve_every_side(native, serve_stream, side):
    """Every side 1..256 at the corner side % 23 (all three rules, masked and not, across the sides)."""
    rs = np.random.RandomState(2000 + side)
    serve_case(native, side, CORNERS[side % len(CORNERS)], rs, serve_stream)


@pytest.mark.parametrize("side", [5, 37, 100, 256])
def test_serve_without_observation_mirror(native, serve_stream, side):
    rs = np.random.RandomState(3000 + side)
    serve_case(native, side, CORNERS[(side + 7) % len(CORNERS)], rs, serve_stream, mirror=False)


# ------------------------------------------------------------------------------------------------------------------
# 3. the facades against OracleEnv: random call interleavings, loads across regimes, the step sequence wrap
# ------------------------------------------------------------------------------------------------------------------
FACADE_SIDES = [1, 3, 33, 100, 256, 257, 274, 275, 300, 448, 449, 480]
FORK_FACADE_SIDES = [3, 100, 257, 300, 449]


def make_facade(CGL, fork, side, corner, seed):
    spawn, smax, rule, empty, emin, _ = corner
    if rule == oracle.DEAD_ZERO:
        env = CGL.sim(side=side, seed=seed, gpu=True, spawnStabilityFactor=spawn, stableStabilityFactor=smax)
        ref = OracleEnv.seeded(side, seed, spawn, smax)
    else:
        env = fork.sim(side=side, seed=seed, gpu=True, spawnStabilityFactor=spawn, stableStabilityFactor=smax,
                       empty=empty, empty_min=emin, dead_rule=RULE_NAME[rule])
        ref = OracleEnv.seeded(side, seed, spawn, smax, rule, empty, emin, masked=True, fork=True)
    return env, ref


class FacadeDriver:
    """Applies one operation to the facade and to its OracleEnv, and checks what the facade returns."""

    def __init__(self, env, ref, rs, live_views):
        self.env, self.ref, self.rs, self.live_views = env, ref, rs, live_views
        self.views = None
        if live_views:
            self.take_views()

    def take_views(self):
        self.views = (self.env.get_state(vector=True, shallow=True), self.env.get_stable(vector=True, shallow=True))

    def check_views(self, what):
        if self.views is not None:
            assert np.array_equal(self.views[0], self.ref.world) and np.array_equal(self.views[1], self.ref.stable), what

    def check_all(self, what):
        env, ref = self.env, self.ref
        assert np.array_equal(env.get_state(vector=True), ref.world), what
        assert np.array_equal(env.get_stable(vector=True), ref.stable), what
        assert int(env.reward()) == ref.reward() and int(env.alive()) == ref.alive(), what
        assert env.get_count() == ref.count, what

    def offers_run(self):
        return self.env._bs.fused or self.env.side <= 274

    def offers_cycle(self):
        return self.env._bs.fused or self.env.side <= 237

    def load_args(self, side, corners):
        """An arbitrary world and int8 plane of `side`, a count and the factors of a random corner of `corners`."""
        rs, size = self.rs, side * side
        corner = corners[rs.randint(len(corners))]
        cells = rs.randint(2, size=size).astype(np.uint8)
        args = [cells, corner_plane(rs, size, corner), side, int(rs.randint(5000)), corner[0], corner[1]]
        if self.ref.fork:
            args.append(corner[3])
        return args

    def do(self, op, what):
        env, ref, rs = self.env, self.ref, self.rs
        side, size = ref.side, ref.size
        if op == "step":
            env.step(); ref.step()
        elif op == "toggle":
            acts = edge_actions(rs, side)
            a = acts[rs.randint(len(acts))]
            a = np.int32(a) if rs.randint(2) else int(a)
            env.toggle_state(a); ref.toggle_state(int(a))
        elif op == "toggle_list":
            idx = [int(v) for v in rs.randint(size, size=int(rs.randint(2, 6)))]
            idx.append(idx[0])                                # a duplicate toggles once
            env.toggle_state(idx); ref.toggle_state(idx)
        elif op == "toggle_noop":
            env.toggle_state([size]); ref.toggle_state([size])
            env.toggle_state(size); ref.toggle_state(size)
        elif op == "dqn":                                     # CGL/main.py:66-71
            acts = edge_actions(rs, side)
            a = np.int32(acts[rs.randint(len(acts))])
            env.toggle_state(a); env.step()
            ref.toggle_state(int(a)); ref.step()
            obs = env.get_stable(vector=True, shallow=self.live_views)
            assert np.array_equal(obs, ref.stable), what
            assert int(env.reward()) == ref.reward(), what
        elif op == "reward":
            assert int(env.reward()) == ref.reward(), what
        elif op == "alive":
            assert int(env.alive()) == ref.alive(), what
        elif op == "state":
            assert np.array_equal(env.get_state(), ref.world.reshape(side, side)), what
        elif op == "stable":
            assert np.array_equal(env.get_stable(), ref.stable.reshape(side, side)), what
        elif op == "reset":
            env.reset(); ref.reset()
        elif op == "match":
            assert env.match(ref.world.reshape(side, side)), what
            other = ref.world.copy()
            other[rs.randint(size)] ^= 1
            assert not env.match(other), what
        elif op == "update":
            new = rs.randint(2, size=size).astype(np.uint8)
            if ref.fork:
                plane = corner_plane(rs, size, CORNERS[rs.randint(len(CORNERS))]) if rs.randint(2) else None
                env.update_state(new.reshape(side, side), plane); ref.update_state(new, plane)
            else:
                env.update_state(new, side); ref.update_state(new)
        elif op == "save":
            sv, want = env.save(), ref.save()
            assert len(sv) == len(want), what
            assert np.array_equal(sv[0], want[0]) and np.array_equal(sv[1], want[1]) and sv[2:] == want[2:], what
            env.load(*sv)
        elif op == "load":
            args = self.load_args(side, FORK_CORNERS if ref.fork else BASE_CORNERS)
            env.load(*args); ref.load(*args)
        elif op == "run":
            if self.offers_run():
                n, fixed = int(rs.randint(1, 8)), bool(rs.randint(4) == 0)
                assert env.run(n, until_fixed=fixed) == ref.run(n, until_fixed=fixed), what
        elif op == "cycle":
            if self.offers_cycle():
                n = int(rs.randint(1, 12))
                assert env.run_until_cycle(n, max_period=2) == ref.run_until_cycle(n, max_period=2), what
        elif op == "action_rewards":
            assert np.array_equal(env.action_rewards(), ref.action_rewards()), what
        else:
            raise ValueError(op)
        if env._pending is None:                              # (a deferred scalar toggle shows once a call applies it)
            self.check_views((what, op))


OPS = ["step"] * 4 + ["dqn"] * 4 + ["toggle"] * 2 + ["toggle_list", "toggle_noop", "reward", "alive", "state", "stable",
                                                      "reset", "match", "update", "save", "load", "run", "cycle",
                                                      "action_rewards"]


def drive(driver, n_ops):
    for it in range(n_ops):
        driver.do(OPS[driver.rs.randint(len(OPS))], it)
    driver.check_all("end")


@pytest.mark.parametrize("live_views", [False, True])
@pytest.mark.parametrize("side", FACADE_SIDES)
def test_facade_random_interleavings(CGL, fork, side, live_views):
    rs = np.random.RandomState(side * 2 + live_views)
    corner = BASE_CORNERS[side % len(BASE_CORNERS)]
    env, ref = make_facade(CGL, fork, side, corner, seed=side)
    drive(FacadeDriver(env, ref, rs, live_views), 90)


@pytest.mark.parametrize("live_views", [False, True])
@pytest.mark.parametrize("side", FORK_FACADE_SIDES)
def test_fork_facade_random_interleavings(CGL, fork, side, live_views):
    rs = np.random.RandomState(side * 3 + live_views)
    corner = FORK_CORNERS[(side + live_views) % len(FORK_CORNERS)]
    env, ref = make_facade(CGL, fork, side, corner, seed=side)
    drive(FacadeDriver(env, ref, rs, live_views), 90)


@pytest.mark.parametrize("linger_us", ["250", "100000"])
@pytest.mark.parametrize("live_views", [False, True])
@pytest.mark.parametrize("facade", ["base", "fork"])
def test_facade_load_across_regimes(CGL, fork, facade, live_views, linger_us, monkeypatch):
    """load() with an arbitrary plane and new factors, right after served or one-launch steps, on the same side and
    across all four regimes: 100 -> 100 -> 300 -> 300 -> 480 -> 64 -> 64 -> 257 -> 3 -> 3.  With the longest linger
    the resident server is still there when load() runs, so load() has to stop it before it writes the planes."""
    monkeypatch.setenv("CGL_SIM_LINGER_US", linger_us)
    rs = np.random.RandomState(17 + live_views + 2 * (facade == "fork"))
    corners = FORK_CORNERS if facade == "fork" else BASE_CORNERS
    env, ref = make_facade(CGL, fork, 100, corners[3], seed=4)
    d = FacadeDriver(env, ref, rs, live_views)
    for i, side in enumerate([100, 300, 300, 480, 64, 64, 257, 3, 3]):
        for op in ("dqn", "dqn", "step", "dqn"):              # the server (or a one-launch step) holds the state now
            d.do(op, (i, side))
        args = d.load_args(side, corners)
        resized = side != ref.side
        env.load(*args); ref.load(*args)
        if live_views and resized:
            d.take_views()                                   # a new side has new mirrors
        d.check_views((i, side, "load"))
        for op in ("dqn", "step", "dqn", "reward", "action_rewards", "stable", "reset", "dqn", "state"):
            d.do(op, (i, side))
        d.check_all((i, side))


@pytest.mark.parametrize("facade", ["base", "fork"])
@pytest.mark.parametrize("side", [100, 300])
def test_facade_step_sequence_wraps(CGL, fork, facade, side):
    """The facade numbers its steps modulo 2^30 (served and one-launch); a loop across the wrap, with the server
    stopped and restarted on both sides of it, returns the oracle's observations."""
    corner = FORK_CORNERS[5] if facade == "fork" else BASE_CORNERS[1]
    env, ref = make_facade(CGL, fork, side, corner, seed=9)
    rs = np.random.RandomState(side)
    d = FacadeDriver(env, ref, rs, live_views=False)
    obs = env.get_stable(vector=True, shallow=True)          # the DQN loop's live observation (the world stays private)
    env._seq = 0x3fffffff - 3
    for i in range(14):
        d.do("dqn", i)
        assert np.array_equal(obs, ref.stable), i
        if i in (2, 6):
            d.do("state", i)                                 # stops the server (QUIT carries a sequence number too)
    assert env._seq < 100                                    # the counter went across the wrap
    d.check_all("end")


# ------------------------------------------------------------------------------------------------------------------
# 4. the host-driven rollout
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("zero_copy", [False, True])
@pytest.mark.parametrize("side", [10, 32, 33, 100, 130, 256])
def test_rollout_matches_oracle_at_base_corners(native, side, zero_copy):
    from cgl_b200.rollout import HostRollout
    size, n_envs, groups = side * side, 6, 2
    per = n_envs // groups
    for ci, corner in enumerate(BASE_CORNERS):
        spawn, smax = corner[:2]
        replicas = 1 + ci % 2
        rs = np.random.RandomState(100 * side + ci)
        ro = HostRollout(n_envs, side, n_groups=groups, n_replicas=replicas, seed=ci, spawnStabilityFactor=spawn,
                         stableStabilityFactor=smax, obs_to_host=True, zero_copy_actions=zero_copy)
        assert ro.zero_copy_actions == zero_copy
        cells = [[None] * replicas for _ in range(groups)]
        stab = [[None] * replicas for _ in range(groups)]
        for g in range(groups):
            for r in range(replicas):
                cells[g][r] = rs.randint(2, size=(per, size)).astype(np.uint8)
                stab[g][r] = np.stack([corner_plane(rs, size, corner) for _ in range(per)])
                sim = ro.sim(g, r)
                sim.set_state(torch.from_numpy(cells[g][r]).cuda())
                sim.stable.copy_(torch.from_numpy(stab[g][r]))
            ro.obs[g][:] = 99
        torch.cuda.synchronize()                             # the rollout's streams do not wait for torch's
        edges = np.array(edge_actions(rs, side), np.int64)
        last_rew = [np.zeros(per, np.int32) for _ in range(groups)]
        log = []

        def pick(rew, step, group):                          # actions that depend on the group's last rewards
            k = (rew.astype(np.int64) * 7 + step * 13 + group * 5 + np.arange(per) * 3) % (2 * edges.size)
            return np.where(k < edges.size, edges[k % edges.size], (rew.astype(np.int64) + k * 31) % (size + 1)
                            ).astype(np.int32)

        def policy(group, step, rewards, actions):
            log.append((group, step))
            actions[:] = pick(rewards, step, group)

        ro.run(5, policy)
        ro.run(2, policy)
        for s in range(7):
            for g in range(groups):
                acts = pick(last_rew[g], s, g)
                rew, _ = oracle.step_batch(cells[g][s % replicas], stab[g][s % replicas], side, acts, spawn, smax)
                last_rew[g] = rew
        assert len(log) == 7 * groups
        for g in range(groups):
            assert np.array_equal(ro.rewards[g], last_rew[g]), (side, corner, g)
            assert np.array_equal(ro.obs[g], stab[g][6 % replicas]), (side, corner, g)
            for r in range(replicas):
                sim = ro.sim(g, r)
                assert np.array_equal(sim.get_state().cpu().numpy(), cells[g][r]), (side, corner, g, r)
                assert np.array_equal(sim.stable.cpu().numpy(), stab[g][r]), (side, corner, g, r)
        ro.close()


# ------------------------------------------------------------------------------------------------------------------
# 5. the host-buffer entry points
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("obs", [False, True])
@pytest.mark.parametrize("side", [10, 33, 64, 100, 256])
def test_env_step_host_matches_oracle(native, side, obs):
    """cgl_env_step_host and cgl_env_step_host_async (alternating), rewards into pinned memory (written by the kernel)
    or into pageable memory (copied), with and without the observation copy."""
    from cgl_b200.batched import BatchedSim
    size, n = side * side, 5
    stream = torch.cuda.Stream()
    for ci, corner in enumerate(BASE_CORNERS):
        spawn, smax = corner[:2]
        rs = np.random.RandomState(10 * side + ci + obs)
        env = BatchedSim(n, side, seed=ci, spawnStabilityFactor=spawn, stableStabilityFactor=smax)
        cells = rs.randint(2, size=(n, size)).astype(np.uint8)
        st = np.stack([corner_plane(rs, size, corner) for _ in range(n)])
        env.set_state(torch.from_numpy(cells).cuda())
        env.stable.copy_(torch.from_numpy(st))
        torch.cuda.synchronize()
        acts_h = torch.empty(n, dtype=torch.int32).pin_memory()
        rew_h = torch.empty(n, dtype=torch.int32)
        rew_h = rew_h.pin_memory() if ci % 2 == 0 else rew_h
        obs_h = torch.empty((n, size), dtype=torch.int8).pin_memory() if obs else None
        edges = edge_actions(rs, side)
        for t in range(4):
            acts = np.array([edges[(t + e) % len(edges)] for e in range(n)], np.int32)
            acts_h.numpy()[:] = acts
            rew_h.fill_(-12345)
            if obs_h is not None:
                obs_h.fill_(99)
            sync = (t + ci) % 2 == 0
            with torch.cuda.stream(stream):
                env.step_host(acts_h, rew_h, obs_h, sync=sync)
                if not sync:
                    env.wait_host()
            rew_o, _ = oracle.step_batch(cells, st, side, acts, spawn, smax)
            what = (side, corner, t, sync)
            assert np.array_equal(rew_h.numpy(), rew_o), what
            if obs_h is not None:
                assert np.array_equal(obs_h.numpy(), st), what
        assert np.array_equal(env.get_state().cpu().numpy(), cells) and np.array_equal(env.stable.cpu().numpy(), st)


@pytest.mark.parametrize("side", [1, 2, 3, 5, 7, 31, 33, 63, 65, 100, 127, 129, 200, 257, 300, 449])
def test_step_state_gpu_matches_oracle(native, side):
    """cgl_step_state_gpu (the reference's __step_state_gpu: host planes in, one step, host planes out) on arbitrary
    planes at every base-rule corner."""
    lib = native.load()
    size = side * side
    rs = np.random.RandomState(side)
    for corner in BASE_CORNERS:
        spawn, smax = corner[:2]
        w = rs.randint(2, size=size).astype(np.uint8)
        s = corner_plane(rs, size, corner)
        cells, st = w.copy(), s.copy()
        for t in range(2):
            native.check(lib.cgl_step_state_gpu(w.ctypes.data, s.ctypes.data, side, spawn, smax), "cgl_step_state_gpu")
            oracle.step(cells, st, side, spawn, smax)
            assert np.array_equal(w, cells) and np.array_equal(s, st), (side, corner, t)
