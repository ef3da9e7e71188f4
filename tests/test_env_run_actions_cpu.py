"""CPU suite: the env run with an action schedule and per-step traces (cgl_env_run_ex).

The host twin restates the bit-sliced run kernel with its toggles and its per-step reward taken from the bit planes
(cgl_bits.cuh sliced_reward32, the very expression the kernel runs); it is checked here against the oracle stepped one
action at a time, every trace row included.  The argument checks of cgl_env_run_ex run before any device work."""
import ctypes
import os

import numpy as np
import pytest

from conftest import PKG, ROOT
from oracle import oracle

TWIN_SRC = os.path.join(ROOT, "tests", "twin", "env_run_actions_twin.cpp")
_lib = None


def _twin():
    """The twin of the traced run kernel, compiled once per session into a temporary directory."""
    global _lib
    if _lib is None:
        import subprocess
        import tempfile
        out = os.path.join(tempfile.mkdtemp(prefix="cgl_run_twin_"), "libenv_run_actions_twin.so")
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", out, TWIN_SRC], check=True)
        L = ctypes.CDLL(out)
        L.twin_env_run_sliced_actions.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32,
                                                  ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                  ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                  ctypes.c_void_p]
        _lib = L
    return _lib


def oracle_run(cells, st, side, acts, spawn, smax, rule, empty, empty_min, masked):
    """One env stepped one action at a time: (reward, alive) after every step; cells / st updated in place."""
    size = side * side
    rew, alv = [], []
    for a in acts:
        a = int(a)
        if 0 <= a < size:
            (oracle.toggle_masked if masked else oracle.toggle)(cells, st, a, spawn)
        oracle.step_rule(cells, st, side, spawn, smax, rule, empty, empty_min)
        rew.append(int(oracle.reward(st)))
        alv.append(int(oracle.alive(cells)))
    return rew, alv


def _schedule(rs, side, k):
    size = side * side
    acts = rs.randint(size, size=k).astype(np.int32)
    acts[rs.rand(k) < 0.2] = size                       # no-ops
    if k > 3:
        acts[2] = acts[1]                               # the same cell twice in a row
    return acts


def _start(rs, side, spawn, empty, rule):
    cells = rs.randint(2, size=side * side).astype(np.uint8)
    st = oracle.initial_stable_fork(cells, spawn, empty) if rule else oracle.initial_stable(cells, spawn)
    return cells, st.astype(np.int8)


def _twin_run(L, cells, st, side, acts, spawn, smax, rule, empty, empty_min, masked, stop=0, k=None):
    k = len(acts) if k is None else k
    words = np.packbits(cells, bitorder="little").view(np.uint32).copy()     # cell j = bit j % 32 of word j // 32
    st = st.copy()
    rew = np.full(k, -7, np.int32)
    alv = np.full(k, 7, np.uint32)
    acts = None if acts is None else np.ascontiguousarray(acts, np.int32)
    rc = L.twin_env_run_sliced_actions(words.ctypes.data, st.ctypes.data, side, k, stop, spawn, smax, rule, empty,
                                       empty_min, int(masked), None if acts is None else acts.ctypes.data,
                                       rew.ctypes.data, alv.ctypes.data)
    out = np.unpackbits(words.view(np.uint8), bitorder="little")
    return out, st, rew, alv, rc & 0xFFFF, rc >> 16


# (spawn, stable_max, empty, empty_min): the defaults, a fork setting, and pairs whose SPAWN..MAX range wraps int8
FACTORS = [(-1, 1, 0, -128), (-2, 2, -1, -5), (5, 127, 0, -128), (100, -100, -3, -20), (3, -128, 2, 10)]


@pytest.mark.parametrize("side", [32, 64, 96, 128, 160, 192, 224, 256])
@pytest.mark.parametrize("rule", [oracle.DEAD_ZERO, oracle.DEAD_DECAY, oracle.DEAD_SAT])
def test_twin_sliced_run_with_actions_equals_oracle_step_by_step(side, rule):
    L = _twin()
    k = 9 if side <= 128 else 5
    for i, (spawn, smax, empty, emin) in enumerate(FACTORS):
        for masked in (False, True):
            rs = np.random.RandomState(side * 31 + rule * 7 + i * 2 + masked)
            cells, st = _start(rs, side, spawn, empty, rule)
            acts = _schedule(rs, side, k)
            got = _twin_run(L, cells, st, side, acts, spawn, smax, rule, empty, emin, masked)
            rew, alv = oracle_run(cells, st, side, acts, spawn, smax, rule, empty, emin, masked)
            what = f"side={side} rule={rule} factors={FACTORS[i]} masked={masked}"
            assert got[4] == k and got[5] == 0, what
            assert np.array_equal(got[0], cells), what
            assert np.array_equal(got[1], st), what
            assert got[2].tolist() == rew, what
            assert got[3].tolist() == alv, what


def test_twin_base_rule_reward_counts_the_wrap_of_planes_loaded_out_of_range():
    # live cells loaded above STABLE (here u = 120 with SPAWN = 5, STABLE = 7): the kernel then takes the wrap term
    L = _twin()
    side, spawn, smax = 64, 5, 7
    rs = np.random.RandomState(3)
    cells, st = _start(rs, side, spawn, 0, 0)
    st[cells != 0] = np.int8(125)
    acts = _schedule(rs, side, 12)
    got = _twin_run(L, cells, st, side, acts, spawn, smax, 0, 0, -128, False)
    rew, alv = oracle_run(cells, st, side, acts, spawn, smax, 0, 0, -128, False)
    assert np.array_equal(got[1], st) and got[2].tolist() == rew and got[3].tolist() == alv


def test_twin_invalid_actions_are_ignored_and_counted():
    L = _twin()
    side, spawn, smax = 32, -1, 1
    rs = np.random.RandomState(8)
    cells, st = _start(rs, side, spawn, 0, 0)
    acts = _schedule(rs, side, 8)
    bad = acts.copy()
    bad[[1, 4, 6]] = [-1, side * side + 1, 1 << 30]
    ok = acts.copy()
    ok[[1, 4, 6]] = side * side
    got = _twin_run(L, cells, st, side, bad, spawn, smax, 0, 0, -128, False)
    rew, alv = oracle_run(cells, st, side, ok, spawn, smax, 0, 0, -128, False)
    assert got[5] == 3
    assert np.array_equal(got[0], cells) and np.array_equal(got[1], st)
    assert got[2].tolist() == rew and got[3].tolist() == alv


def test_twin_traces_under_until_fixed_stop_at_the_fixed_point():
    L = _twin()
    side, spawn, smax, k = 32, -1, 1, 12
    cells = np.zeros(side * side, np.uint8)
    cells[[33, 34, 65, 66]] = 1                         # a block: fixed from the start
    st = oracle.initial_stable(cells, spawn).astype(np.int8)
    got = _twin_run(L, cells, st, side, None, spawn, smax, 0, 0, -128, False, stop=1, k=k)
    assert got[4] == 1
    assert got[2][1:].tolist() == [-7] * (k - 1) and got[3][0] == 4


def test_env_run_ex_rejects_bad_arguments_without_a_gpu():
    import sys
    sys.path.insert(0, PKG)
    from cgl_b200 import native
    lib = native.load()
    w, s, acts, tr_r, tr_a = (ctypes.c_void_p(v).value for v in (0x1000, 0x2000, 0x3000, 0x4000, 0x5000))

    def args(**kw):
        a = native.EnvRunArgs()
        a.world_in, a.world_out, a.stable, a.n_envs, a.side, a.max_steps = w, w, s, 4, 128, 8
        a.spawn, a.stable_max = -1, 1
        for k, v in kw.items():
            setattr(a, k, v)
        return a

    assert lib.cgl_env_run_ex(None, None) == native.E_BADARG
    assert b"null" in lib.cgl_last_error()
    cases = [(dict(world_in=None), b"bad argument"),
             (dict(stable=None), b"bad argument"),
             (dict(n_envs=0), b"bad argument"),
             (dict(side=0), b"bad argument"),
             (dict(n_envs=1 << 31), b"n_envs too large"),
             (dict(dead_rule=3), b"dead_rule"),
             (dict(empty=128), b"int8"),
             (dict(empty_min=-129), b"int8"),
             (dict(masked_toggle=2), b"masked_toggle"),
             (dict(stop_when_fixed=1, actions=acts), b"stop_when_fixed"),
             (dict(reward_trace=tr_r, alive_trace=tr_r), b"separate"),
             (dict(actions=acts, reward_trace=acts), b"separate"),
             (dict(actions=acts, alive_trace=acts), b"separate"),
             (dict(side=275, actions=acts), b"side <= 274")]
    for kw, msg in cases:
        a = args(**kw)
        assert lib.cgl_env_run_ex(ctypes.byref(a), None) == native.E_BADARG, kw
        assert msg in lib.cgl_last_error(), (kw, lib.cgl_last_error())
    # the wrappers share the checks
    assert lib.cgl_env_run_rule(w, w, s, 4, 128, 8, 0, -1, 1, 5, 0, 0, None, None, None, None) == native.E_BADARG
    assert b"dead_rule" in lib.cgl_last_error()
