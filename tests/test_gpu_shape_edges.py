"""GPU suite: every entry point at the shapes where it switches kernels, or where a kernel's index arithmetic meets
the edge of a small grid, bit-exact against the CPU oracle.

  * cgl_life_run around the k-blocked thresholds: cols 928 (not tiled), 960 / 992 (one column group, and a second
    one holding one word), rows 8..33 against K = 2..16 (a torus with fewer rows than K laps more than once per
    launch), chained launches plus a remainder of smaller blocks; torus and open rows;
  * cgl_life_step at its kernel switch (cols 1920 / 4224 generic, 2048 / 4352 streaming) with 1..25 rows,
    1..200 envs, both row modes, with and without live counts;
  * the life kernels' tuning knobs, each forced in a subprocess (the knobs are read once per process), a tuned strip
    length, and RowBandLife on a torus shorter than its kernel_k;
  * the env step at every side 1..300 (generic, byte-plane, fused and > 256 regimes, every side % 4 class), with
    the byte-plane kernel forced on and off, and both dead-cell rules of the CGL_action+ fork;
  * cgl_env_run on arbitrary int8 planes at parameter corners, fused and generic sides up to its side limit,
    each run kernel forced.
The checking functions return or assert on whole shape sets, so that the subprocess variants can import this module
and run the same checks."""
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


def _in_subprocess(knobs, fn):
    """Run fn() of this module in a fresh process with the environment knobs set."""
    script = ("import sys\nsys.path[:0] = sys.argv[1:4]\nimport test_gpu_shape_edges as t\n"
              "getattr(t, sys.argv[4])()\nprint('subprocess ok')\n")
    env = dict(os.environ, **knobs)
    r = subprocess.run([sys.executable, "-c", script, HERE, ROOT, PKG, fn], capture_output=True, text=True, env=env,
                       timeout=900)
    assert r.returncode == 0 and "subprocess ok" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


# ------------------------------------------------------------------------------------------
# life mode
# ------------------------------------------------------------------------------------------
def _pack(cells):
    """uint8 [n, rows, cols] -> packed words on the device (cgl_pack)."""
    native, lib = _native()
    n, rows, cols = cells.shape
    out = torch.empty(n * rows * ((cols + 31) // 32), dtype=torch.int32, device="cuda")
    c = torch.from_numpy(np.ascontiguousarray(cells, np.uint8)).cuda()
    native.check(lib.cgl_pack(native.dptr(c), native.dptr(out), n, rows, cols, native.current_stream()))
    return out


def _unpack(words, n, rows, cols):
    native, lib = _native()
    out = torch.empty(n * rows * cols, dtype=torch.uint8, device="cuda")
    native.check(lib.cgl_unpack(native.dptr(words), native.dptr(out), n, rows, cols, native.current_stream()))
    return out.cpu().numpy().reshape(n, rows, cols)


def _life_open_rows(cells, gens):
    """`gens` generations with dead rows above and below the grid and torus columns (what wrap_rows = 0 means):
    the open window extended by `gens` wrapped columns on each side is exact on its middle columns."""
    cols = cells.shape[1]
    ext = np.concatenate([cells[:, cols - gens:], cells, cells[:, :gens]], axis=1)
    return oracle.life_open(ext, gens)[:, gens:gens + cols]


def _life_run(words, rows, cols, wrap, gens, k):
    native, lib = _native()
    a, b = words.clone(), torch.empty_like(words)
    res = native.ctypes.c_int(-1)
    native.check(lib.cgl_life_run(native.dptr(a), native.dptr(b), rows, cols, wrap, gens, k, native.ctypes.byref(res),
                                  native.current_stream()))
    return a if res.value == 1 else b


def life_run_cases(rows_set, cols_set, ks):
    """cgl_life_run for every (rows, cols, k) and gens in {k, 2k + 3} (chained launches plus a remainder of smaller
    blocks): on the torus the whole grid, with open rows (rows >= 2 gens + 1) the rows at least gens from both
    edges.  Returns the (rows, cols, k, gens, wrap) that differ from the oracle."""
    bad = []
    for rows in rows_set:
        for cols in cols_set:
            cells = np.random.RandomState(rows * 7919 + cols).randint(2, size=(1, rows, cols)).astype(np.uint8)
            words = _pack(cells)
            want = {}
            for k in ks:
                for gens in sorted({k, 2 * k + 3}):
                    for wrap in (1, 0):
                        if not wrap and rows < 2 * gens + 1:
                            continue
                        if (gens, wrap) not in want:
                            want[gens, wrap] = (oracle.life(cells[0], gens, threads=4) if wrap
                                                else _life_open_rows(cells[0], gens)[gens:rows - gens])
                        got = _unpack(_life_run(words, rows, cols, wrap, gens, k), 1, rows, cols)[0]
                        if not np.array_equal(got if wrap else got[gens:rows - gens], want[gens, wrap]):
                            bad.append((rows, cols, k, gens, wrap))
    return bad


def life_step_cases(cols_set, rows_set, envs_set):
    """One cgl_life_step generation of n envs, both row modes, with live counts (written over a dirty buffer) and
    without.  Returns the (cols, rows, n_envs, wrap, counted) that differ from the oracle."""
    native, lib = _native()
    bad = []
    for cols in cols_set:
        for rows in rows_set:
            for n in envs_set:
                cells = np.random.RandomState(cols + 31 * rows + n).randint(2, size=(n, rows, cols)).astype(np.uint8)
                words = _pack(cells)
                for wrap in (1, 0):
                    want = np.stack([oracle.life(c, 1) if wrap else _life_open_rows(c, 1) for c in cells])
                    for counted in (True, False):
                        out = torch.empty_like(words)
                        alive = torch.full((n,), 12345, dtype=torch.int32, device="cuda") if counted else None
                        native.check(lib.cgl_life_step(native.dptr(words), native.dptr(out), n, rows, cols, wrap,
                                                       native.dptr(alive), native.current_stream()))
                        ok = np.array_equal(_unpack(out, n, rows, cols), want)
                        if counted:
                            ok = ok and (alive.cpu().numpy().astype(np.int64) & 0xFFFFFFFF).tolist() == \
                                want.reshape(n, -1).sum(1).tolist()
                        if not ok:
                            bad.append((cols, rows, n, wrap, counted))
    return bad


@pytest.mark.parametrize("cols", [928, 960, 992, 1024, 1952])
def test_life_run_around_k_blocked_thresholds(cuda, cols):
    bad = life_run_cases((8, 9, 11, 12, 13, 15, 16, 17, 24, 33), (cols,), (2, 3, 4, 5, 6, 8, 12, 13, 16))
    assert not bad, f"(rows, cols, k, gens, wrap) that differ from the oracle: {bad}"


@pytest.mark.parametrize("cols", [1920, 2048, 4224, 4352])
def test_life_step_at_kernel_switch(cuda, cols):
    bad = life_step_cases((cols,), (1, 2, 3, 5, 6, 7, 12, 13, 25), (1, 3, 200))
    assert not bad, f"(cols, rows, n_envs, wrap, counted) that differ from the oracle: {bad}"


def variant_life_run():
    bad = life_run_cases((8, 12, 15, 17, 33, 64), (960, 992, 1952), (1, 2, 3, 4, 6, 8, 12, 16))
    assert not bad, f"(rows, cols, k, gens, wrap) that differ from the oracle: {bad}"


def variant_life_step():
    bad = life_step_cases((2048, 4224, 4352), (1, 5, 7, 12, 13, 25, 49), (1, 3, 40))
    assert not bad, f"(cols, rows, n_envs, wrap, counted) that differ from the oracle: {bad}"


@pytest.mark.parametrize("knobs,fn", [
    ({"CGL_TB_CHAIN": "0"}, "variant_life_run"),
    ({"CGL_TB_ROWS": "19"}, "variant_life_run"),         # strips >= K, not a multiple of either unroll
    ({"CGL_LIFE_PF": "6"}, "variant_life_step"),
    ({"CGL_LIFE_MINB": "5"}, "variant_life_step"),
    ({"CGL_LIFE_PDL": "0"}, "variant_life_step"),
    ({"CGL_LIFE_ROWS": "96"}, "variant_life_step"),      # the longest strips (batches of ~19k envs pick them)
], ids=lambda v: ",".join(f"{a}={b}" for a, b in v.items()) if isinstance(v, dict) else v)
def test_life_kernel_variants_at_edges(cuda, knobs, fn):
    _in_subprocess(knobs, fn)


def test_tuned_strip_length_then_run(cuda):
    """cgl_life_tune measures the strip length for (rows, cols, k); the following runs use it."""
    native, lib = _native()
    rows, cols, k = 300, 1984, 8
    cells = np.random.RandomState(1).randint(2, size=(1, rows, cols)).astype(np.uint8)
    words = _pack(cells)
    scratch = torch.empty_like(words)
    native.check(lib.cgl_life_tune(native.dptr(words.clone()), native.dptr(scratch), rows, cols, 1, k,
                                   native.current_stream()))
    for gens in (k, 2 * k + 3):
        got = _unpack(_life_run(words, rows, cols, 1, gens, k), 1, rows, cols)[0]
        assert np.array_equal(got, oracle.life(cells[0], gens, threads=4)), gens


@pytest.mark.parametrize("rows", [8, 12, 16])
def test_row_band_torus_shorter_than_kernel_k(cuda, rows):
    """RowBandLife on one GPU runs the torus through cgl_life_run with k = kernel_k = 16 (16 rows per launch)."""
    from cgl_b200 import bands
    cols = 1024
    cells = np.random.RandomState(rows).randint(2, size=(1, rows, cols)).astype(np.uint8)
    b = bands.RowBandLife(rows, cols, k=16, kernel_k=16)
    b.set_owned(_pack(cells))
    done = 0
    for gens in (16, 19):
        b.run(gens)
        done += gens
        want = oracle.life(cells[0], done)
        assert np.array_equal(_unpack(b.owned.reshape(-1), 1, rows, cols)[0], want), done
        assert b.alive() == int(want.sum())


# ------------------------------------------------------------------------------------------
# env step at every side
# ------------------------------------------------------------------------------------------
# (spawn, stable_max) per side: defaults, int8 extremes both ways round, zero, spawn above max, equal
ENV_FACTORS = ((-2, 2), (-128, 127), (127, -128), (0, 0), (5, 2), (-1, -1))
FUSED = {32, 64, 96, 128, 160, 192, 224, 256}


def env_step_cases(sides, dead_rule="zero", factors=None, empty=0, empty_min=-128, masked=False):
    """Two BatchedSim steps of 3 envs from arbitrary worlds and int8 stability planes, with random actions that
    include the no-op action `size`.  Returns the (side, step) that differ from the oracle."""
    from cgl_b200.batched import DEAD_RULES, BatchedSim
    rule = DEAD_RULES[dead_rule]
    n = 3
    bad = []
    for side in sides:
        spawn, smax = factors or ENV_FACTORS[side % len(ENV_FACTORS)]
        size = side * side
        rs = np.random.RandomState(side * 3 + rule)
        cells = rs.randint(2, size=(n, size)).astype(np.uint8)
        st = rs.randint(-128, 128, size=(n, size)).astype(np.int8)
        env = BatchedSim(n, side, spawnStabilityFactor=spawn, stableStabilityFactor=smax, states=cells,
                         dead_rule=dead_rule, empty=empty, empty_min=empty_min, masked_toggle=masked)
        env.stable.copy_(torch.from_numpy(st))
        for t in range(2):
            acts = rs.randint(size + 1, size=n).astype(np.int32)
            acts[t] = size
            if rule == 0 and not masked:
                rew_o, alv_o = oracle.step_batch(cells, st, side, acts, spawn, smax, threads=4)
            else:
                for e in range(n):
                    if acts[e] < size:
                        (oracle.toggle_masked if masked else oracle.toggle)(cells[e], st[e], int(acts[e]), spawn)
                    oracle.step_rule(cells[e], st[e], side, spawn, smax, rule, empty, empty_min)
                rew_o, alv_o = st.astype(np.int64).sum(1), cells.astype(np.int64).sum(1)
            obs, rew, _ = env.step(torch.from_numpy(acts).cuda(), want_alive=True)
            ok = (np.array_equal(env.get_state().cpu().numpy(), cells) and np.array_equal(obs.cpu().numpy(), st)
                  and rew.cpu().numpy().tolist() == np.asarray(rew_o).tolist()
                  and env.last_alive().cpu().numpy().tolist() == np.asarray(alv_o).tolist())
            if not ok:
                bad.append((side, t))
                break
        env.check_actions()
    return bad


@pytest.mark.parametrize("first", range(1, 301, 30))
def test_env_step_every_side(cuda, first):
    bad = env_step_cases(range(first, first + 30))
    assert not bad, f"(side, step) that differ from the oracle: {bad}"


def variant_env_bytes_forced():
    bad = env_step_cases(range(1, 257))
    assert not bad, f"(side, step) that differ from the oracle: {bad}"


def variant_env_bytes_off():
    bad = env_step_cases([s for s in range(1, 301) if s not in FUSED])
    assert not bad, f"(side, step) that differ from the oracle: {bad}"


@pytest.mark.parametrize("knobs,fn", [({"CGL_ENV_BYTES": "2"}, "variant_env_bytes_forced"),
                                      ({"CGL_ENV_BYTES": "0"}, "variant_env_bytes_off")],
                         ids=["bytes-forced", "bytes-off"])
def test_env_step_every_side_kernel_forced(cuda, knobs, fn):
    _in_subprocess(knobs, fn)


# every regime (generic < 32, byte plane, fused, > 256) and every side % 4 class in each
RULE_SIDES = (1, 2, 3, 4, 7, 10, 31, 32, 33, 34, 35, 36, 64, 99, 128, 131, 198, 255, 256, 257, 258, 259, 260, 300)


@pytest.mark.parametrize("dead_rule", ["decay", "sat"])
def test_env_step_dead_cell_rules_every_side_class(cuda, dead_rule):
    bad = env_step_cases(RULE_SIDES, dead_rule=dead_rule, factors=(127, 127), empty=127, empty_min=-128, masked=True)
    assert not bad, f"(side, step) that differ from the oracle: {bad}"


# ------------------------------------------------------------------------------------------
# cgl_env_run on arbitrary planes
# ------------------------------------------------------------------------------------------
# (dead_rule, spawn, stable_max, empty, empty_min)
RUN_PARAMS = [("zero", -128, 127, 0, -128), ("zero", 127, -128, 0, -128), ("zero", 0, 0, 0, -128),
              ("zero", 5, 2, 0, -128), ("zero", -1, -1, 0, -128),
              ("sat", -2, 2, -128, -128), ("sat", -2, 2, 127, 127), ("sat", -2, 2, 3, -3), ("sat", -2, 2, -1, 127)]
RUN_FUSED_SIDES = (32, 96, 128)
RUN_GENERIC_SIDES = (5, 100, 257, 274)          # 274: the largest side whose three byte planes fit in shared memory


def env_run_cases(params, sides):
    """BatchedSim.run(k) with and without until_fixed, k in {1, 3, 4, 9}, from arbitrary int8 planes; env 0 starts
    empty (fixed after one step), env 1 with one live cell (fixed after two).  Returns the cases that differ."""
    from cgl_b200.batched import DEAD_RULES, BatchedSim
    bad = []
    for dead_rule, spawn, smax, empty, empty_min in params:
        rule = DEAD_RULES[dead_rule]
        for side in sides:
            n, size = (5 if side <= 128 else 3), side * side
            rs = np.random.RandomState(side + 1000 * rule + 7 * (spawn + 128))
            cells0 = rs.randint(2, size=(n, size)).astype(np.uint8)
            cells0[0] = 0
            cells0[1] = 0
            cells0[1, size // 2] = 1
            st0 = rs.randint(-128, 128, size=(n, size)).astype(np.int8)
            env = BatchedSim(n, side, spawnStabilityFactor=spawn, stableStabilityFactor=smax, states=cells0,
                             dead_rule=dead_rule, empty=empty, empty_min=empty_min)
            cells0_d = torch.from_numpy(cells0).cuda()
            for k in (1, 3, 4, 9):
                for until in (False, True):
                    env.set_state(cells0_d)
                    env.stable.copy_(torch.from_numpy(st0))
                    _, rew, steps = env.run(k, until_fixed=until, want_alive=True)
                    cells, st = cells0.copy(), st0.copy()
                    n_o = [oracle.run(cells[e], st[e], side, spawn, smax, k, until_fixed=until) if rule == 0 else
                           oracle.run_rule(cells[e], st[e], side, spawn, smax, k, rule, empty, empty_min,
                                           until_fixed=until) for e in range(n)]
                    ok = (steps.cpu().numpy().tolist() == n_o
                          and np.array_equal(env.get_state().cpu().numpy(), cells)
                          and np.array_equal(env.stable.cpu().numpy(), st)
                          and rew.cpu().numpy().tolist() == st.astype(np.int64).sum(1).tolist()
                          and env.last_alive().cpu().numpy().tolist() == cells.astype(np.int64).sum(1).tolist())
                    if not ok:
                        bad.append((dead_rule, spawn, smax, empty, empty_min, side, k, until))
    return bad


@pytest.mark.parametrize("params", RUN_PARAMS, ids=lambda p: "{}_{}_{}_{}_{}".format(*p))
def test_env_run_parameter_corners(cuda, params):
    bad = env_run_cases([params], RUN_FUSED_SIDES + RUN_GENERIC_SIDES)
    assert not bad, f"(rule, spawn, max, empty, empty_min, side, k, until_fixed) that differ from the oracle: {bad}"


def variant_env_run_fused():
    bad = env_run_cases(RUN_PARAMS, RUN_FUSED_SIDES)
    assert not bad, f"(rule, spawn, max, empty, empty_min, side, k, until_fixed) that differ from the oracle: {bad}"


@pytest.mark.parametrize("impl", ["bytes", "sliced"])
def test_env_run_parameter_corners_kernel_forced(cuda, impl):
    _in_subprocess({"CGL_RUN_IMPL": impl}, "variant_env_run_fused")


def test_env_run_rejects_side_above_shared_memory_limit(cuda):
    from cgl_b200 import native
    from cgl_b200.batched import BatchedSim
    with pytest.raises(native.CglNativeError, match="side <= 274"):
        BatchedSim(1, 275, rng="device").run(1)
