"""CPU suite: ``ssd_step_autoreset`` is exported, ``ssd_episode_end`` matches its ctypes mirror, and NULL or out-of-range
arguments are rejected with SSD_ERR_INVALID before any CUDA call."""
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


def test_symbol_is_exported(lib):
    from homophily_marl_b200 import _capi
    assert hasattr(lib, "ssd_step_autoreset") and "ssd_step_autoreset" in _capi.EXPORTS


def test_episode_end_struct_matches_the_header(tmp_path):
    from homophily_marl_b200 import _capi
    cls = _capi.SsdEpisodeEnd
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "ssd_b200.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(ssd_episode_end));']
    lines += [f'printf("{f} %zu\\n", offsetof(ssd_episode_end, {f}));' for f, _ in cls._fields_]
    lines += ["return 0; }"]
    src = tmp_path / "episode_end.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "episode_end"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["size"]) == C.sizeof(cls) == 24
    for f, _ in cls._fields_:
        assert int(out[f]) == getattr(cls, f).offset, f


def test_bad_arguments_are_rejected_before_any_cuda_call(lib):
    """Without a GPU no handle can be created, so every call here fails validation: a NULL handle, state, actions, `out` or
    `out` member, and bad ranges.  None of them may reach the CUDA runtime."""
    from homophily_marl_b200 import _capi
    before = lib.ssd_last_cuda_error()
    buf = (C.c_uint8 * 256)()
    p = C.cast(buf, C.c_void_p).value
    st = _capi.SsdState(p, p, p, p, p, p)
    so = _capi.SsdStepOut(p, p, p, p, p, p)
    end = _capi.SsdEpisodeEnd(p, p, p)
    acts = C.c_void_p(p)
    call = lambda h, s, a, o, e, lo, cnt: lib.ssd_step_autoreset(h, s, a, None, o, e, lo, cnt, None)  # noqa: E731
    assert call(None, C.byref(st), acts, C.byref(so), C.byref(end), 0, 1) == _capi.SSD_ERR_INVALID
    assert call(None, None, acts, C.byref(so), None, 0, 1) == _capi.SSD_ERR_INVALID
    assert call(None, C.byref(st), None, C.byref(so), None, 0, 1) == _capi.SSD_ERR_INVALID
    assert call(None, C.byref(st), acts, None, None, 0, 1) == _capi.SSD_ERR_INVALID
    for lo, cnt in ((-1, 1), (0, -1), (2 ** 31 - 1, 2)):
        assert call(None, C.byref(st), acts, C.byref(so), None, lo, cnt) == _capi.SSD_ERR_INVALID
    assert lib.ssd_last_cuda_error() == before                 # nothing reached the CUDA runtime


def test_python_layer_accepts_the_new_arguments():
    """The constructor and step_range take the new keywords; the env still refuses to start without a CUDA device."""
    import inspect
    import torch
    from homophily_marl_b200.batch_env import SSDBatchEnv
    assert "keep_episode_end" in inspect.signature(SSDBatchEnv.__init__).parameters
    assert "auto_reset" in inspect.signature(SSDBatchEnv.step_range).parameters
    assert "buf" in inspect.signature(SSDBatchEnv.state_float).parameters
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            SSDBatchEnv("cleanup", 4, 3, map="default3", keep_episode_end=True)
