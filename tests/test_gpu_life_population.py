"""GPU suite: population traces of k-blocked life runs (cgl_life_run_pop, ext.life_run_pop, RowBandLife.run(...,
population=True)), bit-exact against oracle.life stepped one generation at a time.

  * tori at the k-blocked thresholds (rows 8..33 and 1000; cols 928 (not tiled), 960, 992, 1024, 1952, 4096), every
    k, one launch, a remainder and >= 3 chained launches: the trace equals the oracle's populations, and the final
    grid and result_in_a equal the uncounted cgl_life_run;
  * count windows: first row, last row, one row, a window across strip boundaries, and open rows;
  * strip geometry (CGL_TB_ROWS, CGL_TB_CHAIN=0, a tuned strip length), each in a fresh process, and strips longer
    than the counted kernels' 2047-row cap on a dense still life;
  * columns that are not a multiple of 32 (the window count masks the padding bits);
  * row bands: a ring of one through the p2p exchange and LocalBands, against the single torus and alive();
  * the torch extension and its argument checks."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PKG = os.path.join(ROOT, "ecen743-project-cgol_b200")


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from cgl_b200 import native
    native.load()


def _native():
    from cgl_b200 import native
    return native, native.load()


def _pack(cells):
    rows, cols = cells.shape
    bits = cells.reshape(rows, cols // 32, 32).astype(np.uint64)
    words = (bits << np.arange(32, dtype=np.uint64)).sum(-1).astype(np.uint32)
    return torch.from_numpy(words.view(np.int32).reshape(-1)).cuda()


def _unpack(words, rows, cols):
    w = words.cpu().numpy().view(np.uint32).reshape(rows, cols // 32)
    return ((w[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8).reshape(rows, cols)


def _oracle_grids(cells, gens, wrap=True):
    """The grid after each of 1..gens generations (torus, or open rows with torus columns)."""
    out, g = [], cells
    cols = cells.shape[1]
    for _ in range(gens):
        if wrap:
            g = oracle.life(g, 1)
        else:
            ext = np.concatenate([g[:, cols - 1:], g, g[:, :1]], axis=1)
            g = oracle.life_open(ext, 1)[:, 1:1 + cols]
        out.append(g)
    return out


def _run(words, rows, cols, wrap, gens, k, window=None):
    """(final words, result_in_a, trace or None): cgl_life_run, or cgl_life_run_pop with window = (row0, n_rows)."""
    native, lib = _native()
    a, b = words.clone(), torch.empty_like(words)
    res = native.ctypes.c_int(-1)
    st = native.current_stream()
    if window is None:
        native.check(lib.cgl_life_run(native.dptr(a), native.dptr(b), rows, cols, wrap, gens, k,
                                      native.ctypes.byref(res), st), "cgl_life_run")
        pop = None
    else:
        pop = torch.full((gens,), -7, dtype=torch.int64, device="cuda")
        native.check(lib.cgl_life_run_pop(native.dptr(a), native.dptr(b), rows, cols, wrap, gens, k, window[0],
                                          window[1], native.dptr(pop), native.ctypes.byref(res), st), "cgl_life_run_pop")
    torch.cuda.synchronize()
    native.check_alarm()
    return (a if res.value == 1 else b), res.value, (pop.cpu().tolist() if pop is not None else None)


KS = (1, 2, 3, 4, 6, 8, 12, 16)


def _check_tori(shapes, ks=KS):
    """Trace == oracle populations, final grid and result_in_a == uncounted run, for gens in {k, 2k + 3, 3k + 1}."""
    for rows, cols in shapes:
        cells = np.random.RandomState(rows * 7 + cols).randint(2, size=(rows, cols)).astype(np.uint8)
        grids = _oracle_grids(cells, 3 * max(ks) + 3)
        pops = [int(g.sum()) for g in grids]
        words = _pack(cells)
        for k in ks:
            for gens in sorted({k, 2 * k + 3, 3 * k + 1}):
                w1, r1, trace = _run(words, rows, cols, 1, gens, k, (0, rows))
                w0, r0, _ = _run(words, rows, cols, 1, gens, k)
                where = f"rows={rows} cols={cols} k={k} gens={gens}"
                assert trace == pops[:gens], where
                assert r1 == r0 and torch.equal(w1, w0), where
                assert np.array_equal(_unpack(w1, rows, cols), grids[gens - 1]), where


def test_torus_traces_at_the_k_blocked_thresholds(cuda):
    _check_tori([(rows, cols) for rows in (8, 9, 15, 16, 17, 33) for cols in (928, 960, 992, 1024, 1952, 4096)])
    _check_tori([(1000, 960), (1000, 4096)])


def test_count_windows(cuda):
    rows, cols, gens = 1000, 2048, 21
    cells = np.random.RandomState(3).randint(2, size=(rows, cols)).astype(np.uint8)
    grids = _oracle_grids(cells, gens)
    words = _pack(cells)
    for k in (1, 4, 8, 16):
        for row0, n in ((0, 1), (rows - 1, 1), (517, 1), (90, 300), (0, rows), (1, rows - 2)):
            _, _, trace = _run(words, rows, cols, 1, gens, k, (row0, n))
            assert trace == [int(g[row0:row0 + n].sum()) for g in grids], (k, row0, n)
    # open rows: a window at least gens rows from both edges is exact
    rows = 400
    cells = cells[:rows]
    grids = _oracle_grids(cells, gens, wrap=False)
    words = _pack(cells)
    for k in (2, 8, 16):
        for row0, n in ((gens, rows - 2 * gens), (150, 97), (gens, 1)):
            _, _, trace = _run(words, rows, cols, 0, gens, k, (row0, n))
            assert trace == [int(g[row0:row0 + n].sum()) for g in grids], (k, row0, n)


def test_ragged_columns(cuda):
    """cols % 32 != 0: every generation runs as cgl_life_step and the window count masks the padding bits."""
    native, lib = _native()
    rows, cols, gens = 40, 100, 11
    cells = np.random.RandomState(8).randint(2, size=(rows, cols)).astype(np.uint8)
    W = (cols + 31) // 32
    words = torch.empty(rows * W, dtype=torch.int32, device="cuda")
    c = torch.from_numpy(cells).cuda()
    native.check(lib.cgl_pack(native.dptr(c), native.dptr(words), 1, rows, cols, native.current_stream()))
    grids = _oracle_grids(cells, gens)
    for k in (1, 4, 8):
        for row0, n in ((0, rows), (7, 20), (rows - 1, 1)):
            w, _, trace = _run(words, rows, cols, 1, gens, k, (row0, n))
            assert trace == [int(g[row0:row0 + n].sum()) for g in grids], (k, row0, n)
        native.check(lib.cgl_unpack(native.dptr(w), native.dptr(c), 1, rows, cols, native.current_stream()))
        assert np.array_equal(c.cpu().numpy(), grids[-1]), k


def check_strip_geometry():
    """Called in subprocesses with strip knobs set: tori and a window across strips, against the oracle."""
    _check_tori([(1000, 1024), (300, 4096), (33, 992)], ks=(2, 8, 12, 16))
    rows, cols, gens = 1000, 1952, 20
    cells = np.random.RandomState(9).randint(2, size=(rows, cols)).astype(np.uint8)
    grids = _oracle_grids(cells, gens)
    _, _, trace = _run(_pack(cells), rows, cols, 1, gens, 8, (123, 456))
    assert trace == [int(g[123:579].sum()) for g in grids]


def check_strip_cap():
    """Strips longer than 2047 rows (CGL_TB_ROWS=6144) of a dense still life: a thread counts more than 2^16 cells per
    level over such a strip, so the counted kernels must cap their strips (16-bit counts)."""
    rows, cols = 6144, 960
    r, c = np.arange(rows)[:, None], np.arange(cols)[None, :]
    cells = ((r % 3 < 2) & (c % 3 < 2)).astype(np.uint8)         # blocks one cell apart: 4/9 of the cells, stable
    assert np.array_equal(oracle.life(cells, 1), cells)
    live = int(cells.sum())
    words = _pack(cells)
    for k in (4, 8, 16):
        gens = 2 * k + 3
        w, _, trace = _run(words, rows, cols, 1, gens, k, (0, rows))
        assert trace == [live] * gens, k
        assert torch.equal(w, words), k


def check_after_tune():
    native, lib = _native()
    for rows, cols, k in ((1000, 1024, 8), (300, 4096, 16)):
        a = torch.zeros(rows * cols // 32, dtype=torch.int32, device="cuda")
        b = torch.empty_like(a)
        native.check(lib.cgl_life_tune(native.dptr(a), native.dptr(b), rows, cols, 1, k, native.current_stream()))
    check_strip_geometry()


def _in_subprocess(knobs, fn):
    script = ("import sys\nsys.path[:0] = sys.argv[1:4]\nimport test_gpu_life_population as t\n"
              "getattr(t, sys.argv[4])()\nprint('subprocess ok')\n")
    env = dict(os.environ, **knobs)
    r = subprocess.run([sys.executable, "-c", script, HERE, ROOT, PKG, fn], capture_output=True, text=True, env=env,
                       timeout=900)
    assert r.returncode == 0 and "subprocess ok" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


# 100 and 150 leave padding warps at 1000 x 1024 (2 column groups x 10 / 7 strips); 3000: one strip per grid;
# 40 < 8 K turns chaining off for K > 5.
@pytest.mark.parametrize("knobs", [{"CGL_TB_ROWS": "40"}, {"CGL_TB_ROWS": "100"}, {"CGL_TB_ROWS": "150"},
                                   {"CGL_TB_ROWS": "3000"}, {"CGL_TB_CHAIN": "0"}])
def test_strip_geometry_does_not_change_a_count(cuda, knobs):
    _in_subprocess(knobs, "check_strip_geometry")


def test_strips_longer_than_the_count_cap(cuda):
    _in_subprocess({"CGL_TB_ROWS": "6144"}, "check_strip_cap")


def test_counts_after_tuning(cuda):
    _in_subprocess({}, "check_after_tune")


def _bands():
    from cgl_b200 import bands
    return bands


@pytest.mark.parametrize("rows,cols,k,kk,G,gens", [(256, 4096, 16, 8, 2, 37), (512, 2048, 16, 8, 4, 45),
                                                   (96, 2048, 4, 4, 2, 9)])
def test_band_traces_equal_torus_trace(cuda, rows, cols, k, kk, G, gens):
    bands = _bands()
    cells = np.random.RandomState(rows + G).randint(2, size=(rows, cols)).astype(np.uint8)
    words = _pack(cells).view(rows, cols // 32)
    torus = bands.RowBandLife(rows, cols, k=k, kernel_k=kk)
    torus.set_owned(words)
    want = torch.cat([torus.run(gens // 3, population=True), torus.run(gens - gens // 3, population=True)])
    assert want.tolist() == [int(g.sum()) for g in _oracle_grids(cells, gens)]
    assert int(want[-1]) == torus.alive()
    with bands.RowBandLife(rows, cols, k=k, exchange="p2p", kernel_k=kk) as ring:
        ring.set_owned(words)
        got = ring.run(gens, population=True)
        assert torch.equal(got, want) and int(got[-1]) == ring.alive()
        assert torch.equal(ring.owned, torus.owned)
    lb = bands.LocalBands(rows, cols, k, G)
    lb.set_grid(words)
    assert torch.equal(lb.run(gens, population=True), want)
    assert torch.equal(lb.grid(), torus.owned)
    # population=False still returns nothing and runs the same generations
    plain = bands.RowBandLife(rows, cols, k=k, kernel_k=kk)
    plain.set_owned(words)
    assert plain.run(gens) is None and torch.equal(plain.owned, torus.owned)


@pytest.mark.parametrize("exchange", ["p2p", "dist"])
def test_two_gpu_population_trace_equals_single_gpu(cuda, exchange):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tools", "run_bands.py"), "--rows", "4096", "--cols",
           "8192", "--k", "8", "--gens", "43", "--exchange", exchange, "--check", "--population"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert '"ok": true' in r.stdout and '"population_equal": true' in r.stdout


def test_torch_extension_life_run_pop(cuda):
    from cgl_b200 import native
    ext = native.ext()
    rows, cols, gens = 200, 1024, 19
    cells = np.random.RandomState(4).randint(2, size=(rows, cols)).astype(np.uint8)
    grids = _oracle_grids(cells, gens)
    words = _pack(cells)
    for k in (1, 8, 16):
        a, b = words.clone(), torch.empty_like(words)
        pop = torch.empty(gens, dtype=torch.int64, device="cuda")
        in_a = ext.life_run_pop(a, b, rows, cols, True, gens, k, 10, 150, pop)
        a0, b0 = words.clone(), torch.empty_like(words)
        assert in_a == ext.life_run(a0, b0, rows, cols, True, gens, k)
        assert torch.equal(a if in_a else b, a0 if in_a else b0)
        assert pop.tolist() == [int(g[10:160].sum()) for g in grids]
    a, b = words.clone(), torch.empty_like(words)
    good = dict(a=a, b=b, rows=rows, cols=cols, wrap_rows=True, gens=gens, k=8, count_row0=0, count_rows=rows,
                pop=torch.empty(gens, dtype=torch.int64, device="cuda"))
    bad = [dict(pop=torch.empty(gens, dtype=torch.int32, device="cuda")),
           dict(pop=torch.empty(gens, dtype=torch.int64)),
           dict(pop=torch.empty(2 * gens, dtype=torch.int64, device="cuda")[::2]),
           dict(pop=torch.empty(gens + 1, dtype=torch.int64, device="cuda")),
           dict(count_rows=0), dict(count_row0=1), dict(count_row0=-1, count_rows=2)]
    for change in bad:
        with pytest.raises(RuntimeError):
            ext.life_run_pop(**dict(good, **change))
    assert torch.equal(a, words)
