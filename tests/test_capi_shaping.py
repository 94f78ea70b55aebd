"""CPU suite: the shaped-reward surface of the C ABI -- ``ssd_set_reward_shaping`` is declared, exported and bound, the
``ssd_shaping`` layout matches the ctypes mirror, and bad arguments are rejected with SSD_ERR_INVALID before any CUDA call (the
cases that need a handle run on the GPU, in tests/test_gpu_shaping.py)."""
import ctypes as C
import math
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def test_symbol_is_declared_exported_and_bound(lib):
    from homophily_marl_b200 import _capi
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "ssd_b200.h")).read(), flags=re.S)
    assert re.search(r"\bssd_set_reward_shaping\s*\(", text)
    assert hasattr(lib, "ssd_set_reward_shaping") and "ssd_set_reward_shaping" in _capi.EXPORTS
    assert lib.ssd_set_reward_shaping.argtypes[2] is C.POINTER(_capi.SsdShaping)


def test_struct_layout_matches_the_header(tmp_path):
    from homophily_marl_b200 import _capi
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "ssd_b200.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(ssd_shaping));']
    lines += [f'printf("{f} %zu\\n", offsetof(ssd_shaping, {f}));' for f, _ in _capi.SsdShaping._fields_]
    lines += ["return 0; }"]
    src = tmp_path / "shaping.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "shaping"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["size"]) == C.sizeof(_capi.SsdShaping) == 16
    assert [f for f, _ in _capi.SsdShaping._fields_] == ["alpha", "beta", "decay", "prosocial"]
    for f, _ in _capi.SsdShaping._fields_:
        assert int(out[f]) == getattr(_capi.SsdShaping, f).offset, f


def test_bad_arguments_are_rejected_before_any_cuda_call(lib):
    """Without a GPU no handle can be created: every combination below fails validation (a NULL handle at the least) and none
    reaches the CUDA runtime."""
    from homophily_marl_b200 import _capi
    before = lib.ssd_last_cuda_error()
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    good = (_capi.SsdShaping * 2)(_capi.SsdShaping(1.0, 0.5, 0.9, 0.2), _capi.SsdShaping(0.0, 0.0, 1.0, 1.0))
    calls = [(1, good, p, p), (0, None, None, None), (1, good, p, None), (1, good, None, p), (1, None, p, p), (257, good, p, p),
             (-1, good, p, p)]
    for bad in (math.nan, math.inf, -1.0):
        calls += [(1, (_capi.SsdShaping * 1)(_capi.SsdShaping(bad, 0.0, 0.5, 0.0)), p, p)]
    calls += [(1, (_capi.SsdShaping * 1)(_capi.SsdShaping(0.0, 0.0, 1.5, 0.0)), p, p),
              (1, (_capi.SsdShaping * 1)(_capi.SsdShaping(0.0, 0.0, 0.5, -0.5)), p, p)]
    for n, params, trace, shaped in calls:
        assert lib.ssd_set_reward_shaping(None, n, params, trace, shaped) == _capi.SSD_ERR_INVALID, n
    assert lib.ssd_last_cuda_error() == before


def test_python_layer_accepts_the_option():
    import torch
    from homophily_marl_b200.batch_env import SSDBatchEnv
    assert hasattr(SSDBatchEnv, "shaped_reward")
    with pytest.raises(ValueError, match="reward_shaping"):                  # refused before any device is needed
        SSDBatchEnv("cleanup", 4, 3, map="default3", extra_args=dict(reward_shaping={"alpha": 1, "kappa": 2}))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            SSDBatchEnv("cleanup", 4, 3, map="default3", extra_args=dict(reward_shaping={"alpha": 5}))
