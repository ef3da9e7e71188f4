"""GPU suite: row-band life mode.  One GPU: G emulated bands == plain torus == oracle, and a ring of one through the
p2p exchange kernel.  With >= 2 GPUs: torchrun over NVLink with both exchange back ends, checked against the
single-GPU torus."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bands():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200 import bands as b
    return b


def _pack_np(cells):
    rows, cols = cells.shape
    bits = cells.reshape(rows, cols // 32, 32).astype(np.uint64)
    words = (bits << np.arange(32, dtype=np.uint64)).sum(-1).astype(np.uint32)
    return torch.from_numpy(words.view(np.int32))


def _unpack_np(words, rows, cols):
    w = words.cpu().numpy().view(np.uint32).reshape(rows, cols // 32)
    return ((w[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8).reshape(rows, cols)


@pytest.mark.parametrize("rows,cols,k,G,gens", [(256, 4096, 8, 4, 21), (96, 2048, 4, 2, 9), (64, 128, 8, 8, 16)])
def test_emulated_bands_equal_torus_and_oracle(bands, rows, cols, k, G, gens):
    cells = np.random.RandomState(rows + cols).randint(2, size=(rows, cols)).astype(np.uint8)
    words = _pack_np(cells).cuda()
    single = bands.RowBandLife(rows, cols, k=k)
    single.set_owned(words)
    single.run(gens)
    lb = bands.LocalBands(rows, cols, k, G)
    lb.set_grid(words)
    lb.run(gens)
    want = oracle.life(cells, gens, threads=4)
    assert np.array_equal(_unpack_np(single.owned, rows, cols), want)
    assert np.array_equal(_unpack_np(lb.grid(), rows, cols), want)
    assert single.alive() == int(want.sum())


def test_randomize_is_partition_invariant(bands):
    a = bands.RowBandLife(1024, 2048, k=8)
    a.randomize(3)
    parts = []
    for r in range(4):
        b = bands.RowBandLife(1024, 2048, k=8, rank=r, world_size=4, exchange="local")
        b.randomize(3)
        parts.append(b.owned.clone())
    assert torch.equal(torch.cat(parts, 0), a.owned)


@pytest.mark.parametrize("rows,cols,k,kk,runs", [(4096, 8192, 64, 8, (64, 128, 40)), (2048, 4096, 16, 8, (48, 16)),
                                                 (1024, 2048, 8, 4, (8, 24, 4)), (8192, 2048, 32, 16, (96,))])
def test_ring_of_one_with_p2p_exchange_equals_torus(bands, rows, cols, k, kk, runs):
    """exchange="p2p" on ONE rank: the band keeps ghost rows and exchanges with itself through the landing zones
    (cgl_halo_exchange, its upper and lower neighbour being the rank itself) -- every code path of the default
    multi-GPU exchange on one GPU.  Several run() calls in a row (block counters and landing slots carry over);
    compared with the plain torus and, for the small shapes, the CPU oracle."""
    g = torch.Generator(device="cuda"); g.manual_seed(rows + k)
    words = torch.randint(-2 ** 31, 2 ** 31 - 1, (rows, cols // 32), dtype=torch.int32, device="cuda", generator=g)
    torus = bands.RowBandLife(rows, cols, k=k, kernel_k=kk)
    torus.set_owned(words)
    with bands.RowBandLife(rows, cols, k=k, kernel_k=kk, exchange="p2p") as ring:
        assert ring.ghost == k and ring.exchange == "p2p"
        ring.set_owned(words)
        for gens in runs:
            ring.run(gens)
            torus.run(gens)
            assert torch.equal(ring.owned, torus.owned), gens
        assert ring.alive() == torus.alive() and ring.checksum() == torus.checksum()
    if rows * cols <= 2048 * 4096:
        want = oracle.life(_unpack_np(words, rows, cols), sum(runs), threads=8)
        assert np.array_equal(_unpack_np(torus.owned, rows, cols), want)


def test_all_pass_depths_agree(bands):
    """cgl_life_run with k = 2, 4, 8, 16 generations per pass (direct pipeline up to 8, skewed at 16) gives the same
    grid after two consecutive runs."""
    rows, cols = 3000, 4096
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    words = torch.randint(-2 ** 31, 2 ** 31 - 1, (rows, cols // 32), dtype=torch.int32, device="cuda", generator=g)
    outs = []
    for kk in (8, 2, 4, 16):
        b = bands.RowBandLife(rows, cols, k=kk, kernel_k=kk)
        b.set_owned(words)
        b.run(64)
        b.run(32)
        outs.append(b.owned.clone())
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


@pytest.mark.parametrize("exchange", ["p2p", "dist"])
def test_two_gpu_bands_match_single_gpu(bands, exchange):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tools", "run_bands.py"), "--rows", "4096", "--cols",
           "8192", "--k", "8", "--gens", "43", "--exchange", exchange, "--check"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert '"ok": true' in r.stdout
