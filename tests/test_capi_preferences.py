"""CPU suite: the per-agent preference surface of the C ABI -- ``ssd_set_reward_preferences`` is declared, exported and bound,
the ``ssd_preference`` layout matches the ctypes mirror, and bad arguments are rejected with SSD_ERR_INVALID before any CUDA call
(the cases that need a handle run on the GPU, in tests/test_gpu_preferences.py)."""
import ctypes as C
import math
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["alpha", "beta", "decay", "prosocial", "svo_angle", "svo_weight"]


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def test_symbol_is_declared_exported_and_bound(lib):
    from homophily_marl_b200 import _capi
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "ssd_b200.h")).read(), flags=re.S)
    assert re.search(r"\bssd_set_reward_preferences\s*\(", text)
    assert hasattr(lib, "ssd_set_reward_preferences") and "ssd_set_reward_preferences" in _capi.EXPORTS
    assert lib.ssd_set_reward_preferences.argtypes[2] is C.POINTER(_capi.SsdPreference)
    assert len(lib.ssd_set_reward_preferences.argtypes) == 7
    assert lib.ssd_abi_version() == 2


def test_struct_layout_matches_the_header(tmp_path):
    from homophily_marl_b200 import _capi
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "ssd_b200.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(ssd_preference));']
    lines += [f'printf("{f} %zu\\n", offsetof(ssd_preference, {f}));' for f, _ in _capi.SsdPreference._fields_]
    lines += ["return 0; }"]
    src = tmp_path / "preference.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "preference"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["size"]) == C.sizeof(_capi.SsdPreference) == 24
    assert [f for f, _ in _capi.SsdPreference._fields_] == FIELDS
    for f, _ in _capi.SsdPreference._fields_:
        assert int(out[f]) == getattr(_capi.SsdPreference, f).offset, f


def bad_calls():
    """(n_sets, sets, n_rows, set_of, trace, shaped) combinations a handle refuses.  Each is wrong in exactly one way against
    the good call (2, good, 1, roster, p, p)."""
    from homophily_marl_b200 import _capi
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    P = _capi.SsdPreference
    good = (P * 2)(P(1.0, 0.5, 0.9, 0.2, 0.5, 1.0), P(0.0, 0.0, 1.0, 1.0, -3.14159274, 0.0))
    roster = (C.c_uint8 * (16 * 256))(*([1, 0] * (8 * 256)))
    over = (C.c_uint8 * (16 * 256))(*([2] * (16 * 256)))          # an entry >= n_sets
    calls = [(2, good, 1, None, p, p), (2, good, 1, over, p, p), (2, None, 1, roster, p, p), (2, good, -1, roster, p, p),
             (2, good, 257, roster, p, p), (257, good, 1, roster, p, p), (-1, good, 1, roster, p, p),
             (0, None, 1, roster, None, None), (2, good, 1, roster, p, None), (2, good, 1, roster, None, p),
             (2, good, 1, roster, None, None), (0, None, 0, None, p, p)]
    fields = {"alpha": (math.nan, -1.0, math.inf), "beta": (-0.5, math.nan), "decay": (1.5, -0.1, math.nan),
              "prosocial": (1.01, -1.0), "svo_angle": (3.1416, -3.1416, math.inf, math.nan), "svo_weight": (-0.1, math.inf, math.nan)}
    for f, vals in fields.items():
        for v in vals:
            q = dict(zip(FIELDS, (1.0, 0.5, 0.9, 0.2, 0.5, 1.0)))
            q[f] = v
            calls.append((1, (P * 1)(P(**q)), 0, None, p, p))
    return calls


def test_bad_arguments_are_rejected_before_any_cuda_call(lib):
    """Without a GPU no handle can be created: every combination below fails validation (a NULL handle at the least) and none
    reaches the CUDA runtime."""
    from homophily_marl_b200 import _capi
    before = lib.ssd_last_cuda_error()
    for args in bad_calls():
        assert lib.ssd_set_reward_preferences(None, *args) == _capi.SSD_ERR_INVALID, args[:4]
    assert lib.ssd_last_cuda_error() == before
