"""CPU suite: the C-ABI library loads and exports every symbol include/cgl_b200.h declares; the
host facade validates arguments like the reference before it touches a device; no compute calls."""
import json
import os
import re

import numpy as np
import pytest

from conftest import PKG, ROOT

API = json.load(open(os.path.join(ROOT, "tests", "golden", "golden_api.json")))


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "cgl_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(cgl_[a-z0-9_]+)\s*\(", hdr)))


def test_header_symbols_are_exported_and_bound_at_abi_version_2():
    from cgl_b200 import native
    lib = native.load()
    syms = _declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/cgl_b200.h but not exported"
        assert s in native.SIGNATURES, f"{s} has no ctypes signature in native.py"
    assert sorted(native.SIGNATURES) == syms
    assert lib.cgl_abi_version() == 2
    assert lib.cgl_words_per_row(1) == 1 and lib.cgl_words_per_row(32) == 1 and lib.cgl_words_per_row(33) == 2
    assert lib.cgl_env_step_is_fused(128) == 1 and lib.cgl_env_step_is_fused(100) == 0
    assert lib.cgl_env_step_launches(128, 1) == 1 and lib.cgl_env_step_launches(10, 1) == 3


def test_library_is_in_tree_and_has_sm100a_code():
    from cgl_b200 import native
    assert os.path.dirname(native.LIB_PATH) == PKG
    blob = open(native.LIB_PATH, "rb").read()
    assert b"sm_100a" in blob


def test_bad_arguments_are_reported_without_a_gpu():
    from cgl_b200 import native
    lib = native.load()
    assert lib.cgl_pack(None, None, 0, 0, 0, None) == native.E_BADARG
    assert b"cgl_pack" in lib.cgl_last_error()
    with pytest.raises(native.CglNativeError):
        native.check(lib.cgl_env_step(None, None, None, 1, 8, None, -1, 1, None, None, None, None), "cgl_env_step")
    # the resident single-env server refuses misaligned mailboxes and sides it cannot hold before touching the device
    import ctypes
    a = native.SimStepArgs()
    a.world_a = a.world_b = a.stable = 0x1000
    a.side, a.obs_mirror, a.result = 64, 0x2000, 0x3004
    assert lib.cgl_sim_serve(ctypes.byref(a), 0x4000, 0, 1, 100, None) == native.E_BADARG and b"aligned" in lib.cgl_last_error()
    a.result, a.side = 0x3000, 257
    assert lib.cgl_sim_serve(ctypes.byref(a), 0x4000, 0, 1, 100, None) == native.E_BADARG and b"side" in lib.cgl_last_error()
    assert lib.cgl_sim_serve_max_side() == 256


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no CPU fallback", ""), f"{f} mentions the oracle"


@pytest.fixture()
def cgl_module(monkeypatch):
    monkeypatch.delenv("GPU_CAPABLE", raising=False)
    import importlib
    import CGL
    return importlib.reload(CGL)


@pytest.mark.parametrize("kwargs,key", [
    (dict(side="3"), "ctor_side_str"), (dict(side=0), "ctor_side_0"), (dict(seed=-1), "ctor_seed_neg"),
    (dict(seed=1.5), "ctor_seed_float"), (dict(warp=-1), "ctor_warp_neg"),
    (dict(spawnStabilityFactor=1.0), "ctor_spawn_float"), (dict(stableStabilityFactor=1.0), "ctor_stable_float"),
    (dict(state=(1, 0)), "ctor_state_tuple"), (dict(state=np.zeros(0)), "ctor_state_empty"),
    (dict(spawnStabilityFactor=-200), "ctor_spawn_overflow"),
])
def test_constructor_validation_matches_reference(cgl_module, kwargs, key):
    """Exception classes recorded from the reference (tests/golden/golden_api.json)."""
    import builtins
    exc = getattr(builtins, API[key])
    with pytest.raises(exc):
        cgl_module.sim(gpu=True, **kwargs)


def test_gpu_capable_switch_matches_reference(monkeypatch):
    import importlib
    import CGL
    monkeypatch.setenv("GPU_CAPABLE", "false")
    mod = importlib.reload(CGL)
    with pytest.raises(TypeError):           # GPU_CAPABLE=false vs gpu=True (CGL/CGL.py:81-82)
        mod.sim(gpu=True)
    with pytest.raises(RuntimeError):        # equal, but this build has no CPU step
        mod.sim(gpu=False)
    monkeypatch.setenv("GPU_CAPABLE", "maybe")
    with pytest.raises(TypeError):
        importlib.reload(CGL)
    monkeypatch.delenv("GPU_CAPABLE")
    importlib.reload(CGL)


def test_no_cpu_fallback_without_a_device(cgl_module):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from cgl_b200 import native
    with pytest.raises(native.CglNativeError):
        cgl_module.sim(side=8, gpu=True)
    from cgl_b200.batched import BatchedSim
    with pytest.raises(native.CglNativeError):
        BatchedSim(2, 8, device="cpu")
