"""GPU suite: env state planes in hardware-compressed device memory (cgl_state_alloc, BatchedSim(_compressed_planes=)).

Compression changes only how the L2 stores lines in DRAM, so a compressed batch must compute exactly what a plain one
computes, on any plane contents, in every way a batch is stepped; creating and deleting batches must not leak device memory;
and batches too small for one allocation granule stay in plain memory."""
import pytest
import torch

pytestmark = pytest.mark.gpu

B_C2, SIDE = 4096, 128
BOTH = ("world", "stable")


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200 import native
    native.load()
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def granularity(cuda):
    from cgl_b200 import native
    g = int(native.load().cgl_state_granularity(0))
    if not g:
        pytest.skip("this device or driver does not offer compressible memory "
                    "(CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED is 0)")
    return g


def _sim(cuda, B, seed, planes, side=SIDE):
    from cgl_b200.batched import BatchedSim
    return BatchedSim(B, side, seed=seed, spawnStabilityFactor=-2, stableStabilityFactor=2, device=cuda, rng="device",
                      _compressed_planes=planes)


def _scramble(sims, seed):
    """Arbitrary contents: uniform random int8 stability (dead cells included) and random world bits."""
    g = torch.Generator(device=sims[0].device)
    for i, s in enumerate(sims):
        g.manual_seed(seed + i)
        s.stable.copy_(torch.randint(-128, 128, s.stable.shape, dtype=torch.int8, device=s.device, generator=g))
        s._wa.copy_(torch.randint(-2 ** 31, 2 ** 31 - 1, s._wa.shape, dtype=torch.int32, device=s.device, generator=g))


def _pair(cuda, n, B=1024):
    """n compressed and n plain batches with the same seeds and the same arbitrary planes."""
    comp = [_sim(cuda, B, 100 * i, BOTH) for i in range(n)]
    plain = [_sim(cuda, B, 100 * i, ()) for i in range(n)]
    _scramble(comp, 7)
    _scramble(plain, 7)
    for s in comp:
        assert all(s.compressed_planes().values()), s.compressed_planes()
    for s in plain:
        assert not any(s.compressed_planes().values())
    return comp, plain


def _assert_same(comp, plain):
    torch.cuda.synchronize()
    for c, p in zip(comp, plain):
        assert torch.equal(c._wa, p._wa)
        assert torch.equal(c.stable, p.stable)
        assert torch.equal(c._reward, p._reward)


def test_c2_planes_are_compressed(cuda, granularity):
    from cgl_b200.batched import COMPRESSED_PLANES
    s = _sim(cuda, B_C2, 0, None)
    got = s.compressed_planes()
    assert got == {"world_a": "world" in COMPRESSED_PLANES, "world_b": "world" in COMPRESSED_PLANES,
                   "stable": "stable" in COMPRESSED_PLANES}
    assert s.stable.numel() >= granularity


def _actions(cuda, B, n=16, seed=5):
    g = torch.Generator(device=cuda)
    g.manual_seed(seed)
    return torch.randint(0, SIDE * SIDE + 1, (n, B), dtype=torch.int32, device=cuda, generator=g)


def test_eager_step_sequence_matches_plain(cuda, granularity):
    from cgl_b200.batched import StepSequence
    comp, plain = _pair(cuda, 2)
    acts = _actions(cuda, comp[0].n_envs)
    for sims in (comp, plain):
        StepSequence(sims, acts).run(64)
    _assert_same(comp, plain)


def test_graph_replay_matches_plain(cuda, granularity):
    from cgl_b200.batched import StepSequence
    comp, plain = _pair(cuda, 2)
    acts = _actions(cuda, comp[0].n_envs)
    for sims in (comp, plain):
        seq = StepSequence(sims, acts)
        seq.run(4)                                          # warm-up outside the capture: planes back in place
        torch.cuda.synchronize()
        stream, graph = torch.cuda.Stream(device=cuda), torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            with torch.cuda.graph(graph, stream=stream):
                seq.run(4)
        for _ in range(15):                                 # 4 + 60 steps
            graph.replay()
    _assert_same(comp, plain)


def test_step_into_caller_buffers_matches_plain(cuda, granularity):
    (c,), (p,) = _pair(cuda, 1)
    acts = _actions(cuda, c.n_envs)
    bufs = {s: [torch.empty_like(s.stable) for _ in range(2)] for s in (c, p)}
    for t in range(64):
        for s in (c, p):
            s.step(acts[t % 16], obs_out=bufs[s][t % 2])
        assert torch.equal(c._reward, p._reward)
    assert c.compressed_planes()["stable"] is False         # the caller's buffer is the observation now
    _assert_same([c], [p])


def test_creating_and_deleting_c2_batches_leaks_nothing(cuda, granularity):
    def cycle():
        s = _sim(cuda, B_C2, 0, None)
        torch.cuda.synchronize()
        del s
        torch.cuda.empty_cache()

    cycle()                                                 # the first batch may leave cached blocks in the pool
    free0, _ = torch.cuda.mem_get_info(cuda)
    for _ in range(20):
        cycle()
    free1, _ = torch.cuda.mem_get_info(cuda)
    plane_bytes = B_C2 * SIDE * SIDE * 1.25
    assert abs(free1 - free0) < plane_bytes, (free0, free1)


@pytest.mark.parametrize("B, side", [(1, 8), (64, 32), (8, 128)])
def test_small_batches_stay_plain(cuda, B, side):
    from cgl_b200 import native
    s = _sim(cuda, B, 0, BOTH, side=side)
    g = int(native.load().cgl_state_granularity(0))
    assert s.stable.numel() < g or not g
    assert not any(s.compressed_planes().values())
