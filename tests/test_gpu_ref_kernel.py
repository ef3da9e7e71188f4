"""GPU suite: our kernels against the REFERENCE's OWN CUDA kernels executing on the same GPU.

The cubins under tests/golden/ref_kernels/ are the kernel strings of /root/reference/CGL/CGL.py:146-182 (base env)
and /root/reference/CGL/CGL_action+/CGL.py:159-196 (fork) compiled for sm_100a by tests/golden/make_ref_cubins.py;
oracle/ref_gpu.py launches them exactly as the reference does (block 256, grid ceil(size/256)).  Nothing here reads
/root/reference.

This is what pins the fork's CUDA-kernel rule ("decay": dead cells fall by one per step to empty_min, :190-193) BY
EXECUTION -- the fork's CPU step (:256) computes something else, so recorded CPU traces cannot pin it -- and it
cross-checks the base rule a second way (the golden traces come from the reference's CPU loop, these results from its
GPU kernel).  Bit-exact on world and stability, every step.
"""
import numpy as np
import pytest

from conftest import FORK_TRACES, TRACES
from oracle import oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    pytest.importorskip("cuda.bindings.driver")
    from oracle import ref_gpu as mod
    return mod


@pytest.fixture(scope="module")
def B():
    from cgl_b200.batched import BatchedSim
    return BatchedSim


class RefEnvs:
    """n independent envs stepped by the reference kernel (one launch per env, like n `sim` objects)."""

    def __init__(self, kernel, cells, stable, side):
        self.k, self.side = kernel, side
        self.world = torch.from_numpy(np.ascontiguousarray(cells, dtype=np.uint8)).cuda()
        self.result = torch.empty_like(self.world)
        self.stable = torch.from_numpy(np.ascontiguousarray(stable, dtype=np.int8)).cuda()

    def step(self):
        for e in range(self.world.shape[0]):
            self.k.step_tensors(self.world[e], self.result[e], self.stable[e], self.side)
        self.world, self.result = self.result, self.world

    def toggle(self, acts, spawn, masked):
        """toggle_state for one index per env (CGL/CGL.py:322-328; fork CGL_action+/CGL.py:377-384)."""
        size = self.side * self.side
        for e, a in enumerate(acts):
            a = int(a)
            if a == size:
                continue
            self.world[e, a] ^= 1
            self.stable[e, a] = spawn * int(self.world[e, a]) if masked else spawn

    def host(self):
        return self.world.cpu().numpy(), self.stable.cpu().numpy()


def random_planes(rs, n, side, binary_stable_range=(-128, 128)):
    size = side * side
    cells = (rs.random_sample((n, size)) < rs.uniform(0.2, 0.6)).astype(np.uint8)
    stable = rs.randint(*binary_stable_range, size=(n, size)).astype(np.int8)
    return cells, stable


BASE_SETS = [(1, -1), (2, -2), (3, -2), (4, -3), (127, -128), (2, 5)]           # (stable_max, spawn)
FORK_SETS = [(2, -128, -2), (2, -5, -2), (2, -6, -2), (2, 7, -2), (3, -6, -1), (3, -6, 0), (4, -90, -3),
             (127, -128, -128)]                                                  # (stable_max, empty_min, spawn)


@pytest.mark.parametrize("consts", BASE_SETS)
@pytest.mark.parametrize("side", [1, 2, 3, 5, 10, 32, 33, 64, 96, 128, 200])
def test_base_rule_equals_reference_cuda_kernel(ref_gpu, B, consts, side):
    stable_max, spawn = consts
    n, size = 3, side * side
    rs = np.random.RandomState(side * 7 + stable_max)
    cells, stable = random_planes(rs, n, side)
    ref = RefEnvs(ref_gpu.RefKernel("base", stable_max, spawn), cells, stable, side)
    env = B(n, side, spawnStabilityFactor=spawn, stableStabilityFactor=stable_max, states=cells)
    env.stable.copy_(torch.from_numpy(stable))
    oc, os_ = cells.copy(), stable.copy()
    for t in range(6):
        acts = rs.randint(size + 1, size=n).astype(np.int32)
        ref.toggle(acts, spawn, masked=False)
        ref.step()
        obs, rew, _ = env.step(torch.from_numpy(acts).cuda())
        oracle.step_batch(oc, os_, side, acts, spawn, stable_max, threads=1)
        rw, rs_ = ref.host()
        assert np.array_equal(env.get_state().cpu().numpy(), rw), (side, consts, t)
        assert np.array_equal(obs.cpu().numpy(), rs_), (side, consts, t)
        assert np.array_equal(oc, rw) and np.array_equal(os_, rs_), ("oracle", side, consts, t)
        assert np.array_equal(rew.cpu().numpy(), rs_.astype(np.int32).sum(axis=1))


@pytest.mark.parametrize("consts", FORK_SETS)
@pytest.mark.parametrize("side", [1, 2, 5, 10, 32, 33, 64, 128, 160])
def test_decay_rule_equals_fork_cuda_kernel(ref_gpu, B, consts, side):
    """dead_rule="decay" (the fork facade's default) against the fork's CUDA kernel: fused step, generic step,
    the on-chip run kernels and the CPU oracle's restatement, on arbitrary int8 planes with masked toggles."""
    stable_max, empty_min, spawn = consts
    n, size = 3, side * side
    rs = np.random.RandomState(side * 11 + stable_max - empty_min)
    cells, stable = random_planes(rs, n, side)
    ref = RefEnvs(ref_gpu.RefKernel("fork", stable_max, spawn, empty_min), cells, stable, side)
    kw = dict(spawnStabilityFactor=spawn, stableStabilityFactor=stable_max, states=cells, dead_rule="decay", empty=-1,
              empty_min=empty_min, masked_toggle=True)
    env = B(n, side, **kw)
    env.stable.copy_(torch.from_numpy(stable))
    oc, os_ = cells.copy(), stable.copy()
    for t in range(6):
        acts = rs.randint(size + 1, size=n).astype(np.int32)
        ref.toggle(acts, spawn, masked=True)
        ref.step()
        obs, rew, _ = env.step(torch.from_numpy(acts).cuda())
        for e in range(n):
            if acts[e] < size:
                oracle.toggle_masked(oc[e], os_[e], int(acts[e]), spawn)
            oracle.step_rule(oc[e], os_[e], side, spawn, stable_max, oracle.DEAD_DECAY, -1, empty_min)
        rw, rs_ = ref.host()
        assert np.array_equal(env.get_state().cpu().numpy(), rw), (side, consts, t)
        assert np.array_equal(obs.cpu().numpy(), rs_), (side, consts, t)
        assert np.array_equal(oc, rw) and np.array_equal(os_, rs_), ("oracle", side, consts, t)
    # plain multi-step runs (cgl_env_run_rule: byte kernel for k < 4, bit-sliced decay kernel from k = 4 on)
    if side <= 274:
        for k in (3, 9):
            for _ in range(k):
                ref.step()
            env.run(k)
            rw, rs_ = ref.host()
            assert np.array_equal(env.get_state().cpu().numpy(), rw), (side, consts, "run", k)
            assert np.array_equal(env.stable.cpu().numpy(), rs_), (side, consts, "run", k)


@pytest.mark.parametrize("name", sorted(FORK_TRACES))
def test_fork_facade_default_rule_follows_fork_cuda_kernel(ref_gpu, name):
    """The CGL_action+ facade (default dead_rule="decay") driven by the recorded fork actions from the recorded
    initial state, against the fork's CUDA kernel stepping the same state: what `CGL_action+/CGL.py` with gpu=True
    computes."""
    import importlib.util
    import os
    from conftest import PKG
    tr = FORK_TRACES[name]
    if not ref_gpu.available("fork", tr.stable_max, tr.spawn, tr.empty_min):
        pytest.skip("no cubin for these constants")
    spec = importlib.util.spec_from_file_location("cgl_fork_facade_ref", os.path.join(PKG, "CGL_action+", "CGL.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    env = mod.sim(state=tr.worlds[0].reshape(tr.side, tr.side), gpu=True, spawnStabilityFactor=tr.spawn,
                  stableStabilityFactor=tr.stable_max, empty=tr.empty, empty_min=tr.empty_min)
    assert np.array_equal(env.get_stable(vector=True), tr.stables[0])           # initial plane: pinned by the trace
    ref = RefEnvs(ref_gpu.RefKernel("fork", tr.stable_max, tr.spawn, tr.empty_min), tr.worlds[0][None, :],
                  tr.stables[0][None, :], tr.side)
    for t in range(tr.T):
        a = tr.actions[t]
        a = [int(v) for v in a[a >= 0]]
        if a:
            env.toggle_state(a if len(a) > 1 else np.int32(a[0]))
            for idx in dict.fromkeys(a):                                         # duplicates toggle once
                ref.toggle([idx], tr.spawn, masked=True)
        env.step()
        ref.step()
        rw, rs_ = ref.host()
        assert np.array_equal(env.get_state(vector=True), rw[0]), (name, t)
        assert np.array_equal(env.get_stable(vector=True), rs_[0]), (name, t)
        assert int(env.stability()) == int(rs_[0].astype(np.int32).sum())


@pytest.mark.parametrize("name", ["rand64_actions", "blinker5", "wrap6", "multi10", "tiny33", "pulsar25", "env128_0"])
def test_reference_cuda_kernel_reproduces_reference_cpu_traces(ref_gpu, name):
    """Sanity of the fixture itself: the reference's GPU kernel replays traces recorded from the reference's CPU
    loop (the two back ends of CGL/CGL.py agree for the base env)."""
    tr = TRACES[name]
    if not ref_gpu.available("base", tr.stable_max, tr.spawn):
        pytest.skip("no cubin for these constants")
    ref = RefEnvs(ref_gpu.RefKernel("base", tr.stable_max, tr.spawn), tr.worlds[0][None, :], tr.stables[0][None, :],
                  tr.side)
    for t in range(tr.T):
        a = tr.action(t)
        if a is not None:
            for idx in dict.fromkeys([a] if isinstance(a, int) else a):
                ref.toggle([idx], tr.spawn, masked=False)
        ref.step()
        rw, rs_ = ref.host()
        assert np.array_equal(rw[0], tr.worlds[t + 1]) and np.array_equal(rs_[0], tr.stables[t + 1]), (name, t)
