"""CPU suite: population traces of RowBandLife / LocalBands, and the argument checks of cgl_life_run_pop.

As in test_bands_cpu.py the stepping function is the host twin of the product's bit logic; here the counted block
`bands._life_block_pop` is swapped for a twin that also popcounts the count window after every generation.  What is
tested is the product's window arithmetic: which rows each band counts, how blocks of kb generations fill their
slice of the trace, and the one all_reduce over the ranks."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import PKG, ROOT
from oracle import oracle
from test_bands_cpu import _grid, _twin


def _cpu_pop_factory():
    L = _twin()

    def block(lib, a, b, rows, cols, wrap_rows, gens, k, count_row0, count_rows, pop, stream):
        assert pop.dtype == torch.int64 and pop.numel() == gens
        W = cols // 32
        src, dst = a, b
        for i in range(gens):
            L.twin_life_generic(src.data_ptr(), dst.data_ptr(), 1, rows, cols, wrap_rows)
            win = dst[count_row0 * W:(count_row0 + count_rows) * W].numpy().view(np.uint32)
            pop[i] = int(np.unpackbits(win.view(np.uint8)).sum())
            src, dst = dst, src
        return src is a
    return block


def _oracle_trace(cells, gens):
    out, g = [], cells
    for _ in range(gens):
        g = oracle.life(g, 1)
        out.append(int(g.sum()))
    return out


def _worker(rank, world, port, rows, cols, k, kernel_k, gens, out_dir):
    sys.path.insert(0, PKG)
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from cgl_b200 import bands
    bands._life_block_pop = _cpu_pop_factory()
    _, words = _grid(rows, cols, 11)
    b = bands.RowBandLife(rows, cols, k=k, rank=rank, world_size=world, device="cpu", exchange="dist",
                          kernel_k=kernel_k)
    b.set_owned(words[rank * b.band_rows:(rank + 1) * b.band_rows])
    first = b.run(gens // 2, population=True)
    second = b.run(gens - gens // 2, population=True)
    torch.save(torch.cat([first, second]), os.path.join(out_dir, f"pop{rank}.pt"))
    torch.save(torch.tensor([b.generation, b.launches]), os.path.join(out_dir, f"gen{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.parametrize("rows,cols,k,kernel_k,gens", [(24, 64, 4, None, 13), (32, 96, 8, 3, 21)])
def test_two_rank_population_trace_equals_oracle(tmp_path, rows, cols, k, kernel_k, gens):
    port = 31500 + (os.getpid() + rows + gens) % 2000
    mp.start_processes(_worker, args=(2, port, rows, cols, k, kernel_k, gens, str(tmp_path)), nprocs=2, join=True,
                       start_method="spawn")
    cells, _ = _grid(rows, cols, 11)
    want = _oracle_trace(cells, gens)
    kk = kernel_k or min(k, 8)
    for r in range(2):
        assert torch.load(os.path.join(tmp_path, f"pop{r}.pt")).tolist() == want       # all-reduced on every rank
        gen, launches = torch.load(os.path.join(tmp_path, f"gen{r}.pt")).tolist()
        assert gen == gens
        blocks = [min(k, n - d) for n in (gens // 2, gens - gens // 2) for d in range(0, n, k)]
        assert launches == sum(-(-kb // kk) for kb in blocks)


def _with_pop_twin(fn):
    sys.path.insert(0, PKG)
    from cgl_b200 import bands
    old_pop, old = bands._life_block_pop, bands._life_block
    bands._life_block_pop = _cpu_pop_factory()
    bands._life_block = lambda *a, **kw: pytest.fail("population=True must not take the uncounted block")
    try:
        return fn(bands)
    finally:
        bands._life_block_pop, bands._life_block = old_pop, old


def test_single_torus_and_local_bands_population_traces_equal_oracle():
    rows, cols, gens = 32, 64, 11
    cells, words = _grid(rows, cols, 5)
    want = _oracle_trace(cells, gens)

    def run(bands):
        single = bands.RowBandLife(rows, cols, k=4, device="cpu")
        single.set_owned(words)
        assert single.run(gens, population=True).tolist() == want
        assert single.generation == gens and single.launches == 3
        for n_bands in (2, 4):
            lb = bands.LocalBands(rows, cols, 4, n_bands, device="cpu")
            lb.set_grid(words)
            assert lb.run(gens, population=True).tolist() == want
        assert single.run(0, population=True).numel() == 0
    _with_pop_twin(run)


def test_life_run_pop_rejects_bad_arguments_without_a_gpu():
    sys.path.insert(0, PKG)
    from cgl_b200 import native
    lib = native.load()
    a, b, pop = ctypes.c_void_p(0x1000), ctypes.c_void_p(0x2000), ctypes.c_void_p(0x3000)
    res = ctypes.c_int(-1)
    cases = [((a, b, 64, 1024, 1, 8, 8, 0, 64, None), b"NULL"),
             ((a, b, 64, 1024, 1, 8, 8, 0, 0, pop), b"count_rows"),
             ((a, b, 64, 1024, 1, 8, 8, 1, 64, pop), b"window"),
             ((a, b, 64, 1024, 1, 8, 8, 64, 1, pop), b"window"),
             ((a, b, 64, 1024, 1, 8, 8, 0xFFFFFFFF, 2, pop), b"window")]
    for args, msg in cases:
        assert lib.cgl_life_run_pop(*args, ctypes.byref(res), None) == native.E_BADARG
        assert msg in lib.cgl_last_error()
        assert res.value == -1
