"""CPU suite: the index4 state entry points of the C ABI -- ``ssd_state_layout`` matches its ctypes mirror, and
``ssd_set_state_format``, ``ssd_get_state_layout`` and ``ssd_expand_state`` reject a NULL handle, an unknown format and NULL
buffers before any CUDA call."""
import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def test_state_layout_struct_matches_the_header(tmp_path):
    from homophily_marl_b200 import _capi
    cls = _capi.SsdStateLayout
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "ssd_b200.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(ssd_state_layout));']
    lines += [f'printf("{f} %zu\\n", offsetof(ssd_state_layout, {f}));' for f, _ in cls._fields_]
    lines += ["return 0; }"]
    src = tmp_path / "state_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "state_layout"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["size"]) == C.sizeof(cls) == 16
    for f, _ in cls._fields_:
        assert int(out[f]) == getattr(cls, f).offset, f


def test_state_entry_points_reject_bad_arguments(lib):
    from homophily_marl_b200 import _capi
    before = lib.ssd_last_cuda_error()
    lay = _capi.SsdStateLayout()
    buf = (C.c_uint8 * 64)()
    out = (C.c_float * 64)()
    for fmt in (_capi.SSD_OBS_RGB, _capi.SSD_OBS_INDEX4, 2, -1):
        assert lib.ssd_get_state_layout(None, fmt, C.byref(lay)) == _capi.SSD_ERR_INVALID
        assert lib.ssd_get_state_layout(None, fmt, None) == _capi.SSD_ERR_INVALID
        assert lib.ssd_set_state_format(None, fmt) == _capi.SSD_ERR_INVALID
    assert lib.ssd_expand_state(None, C.cast(buf, C.c_void_p), 0, 1, C.cast(out, C.c_void_p), None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_expand_state(None, None, 0, 0, None, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_last_cuda_error() == before                 # nothing reached the CUDA runtime


def test_python_rejects_an_unknown_state_format():
    """extra_args["state_format"] is validated before the env touches CUDA."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    with pytest.raises(ValueError, match="state_format"):
        SSDBatchEnv("cleanup", 4, 3, map="default3", extra_args=dict(state_format="rgb8"))
