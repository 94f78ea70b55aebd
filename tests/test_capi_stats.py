"""CPU suite: the episode-counter surface of the C ABI -- ``ssd_set_stats`` is exported, the SSD_STAT_* constants of the header
match the ctypes mirror, and bad arguments are rejected with SSD_ERR_INVALID before any CUDA call (the episode_limit bound needs a
handle, so that case runs on the GPU)."""
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


def test_constants_match_the_header(tmp_path):
    from homophily_marl_b200 import _capi
    names = ["SSD_N_STATS"] + [f"SSD_STAT_{k.upper()}" for k in _capi.STAT_NAMES]
    lines = ['#include <stdio.h>', '#include "ssd_b200.h"', 'int main(void) {']
    lines += [f'printf("{k} %d\\n", {k});' for k in names] + ["return 0; }"]
    src = tmp_path / "stats.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "stats"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert {k: int(v) for k, v in out.items()} == {k: getattr(_capi, k) for k in names}
    assert _capi.SSD_N_STATS == 7 and list(range(7)) == [getattr(_capi, k) for k in names[1:]]


def test_symbol_is_exported(lib):
    from homophily_marl_b200 import _capi
    assert hasattr(lib, "ssd_set_stats") and "ssd_set_stats" in _capi.EXPORTS


def test_bad_arguments_are_rejected_before_any_cuda_call(lib):
    """Without a GPU no handle can be created: a NULL handle, and end_stats without stats, fail validation.  None of these calls
    may reach the CUDA runtime."""
    from homophily_marl_b200 import _capi
    before = lib.ssd_last_cuda_error()
    buf = (C.c_uint32 * 64)()
    p = C.cast(buf, C.c_void_p)
    assert lib.ssd_set_stats(None, p, p) == _capi.SSD_ERR_INVALID
    assert lib.ssd_set_stats(None, p, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_set_stats(None, None, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_set_stats(None, None, p) == _capi.SSD_ERR_INVALID
    assert lib.ssd_last_cuda_error() == before


@pytest.mark.gpu
def test_episode_limit_bound_and_end_stats_without_stats_on_a_handle(lib):
    """episode_limit 65 536 is refused (APPLE_T of an episode must stay below 2^31), 65 535 accepted; end_stats without stats is
    refused on a real handle too; NULL, NULL always turns counting off.  The refusals happen before any CUDA call."""
    import torch
    from homophily_marl_b200 import _capi
    from homophily_marl_b200.batch_env import SSDBatchEnv
    buf = torch.zeros(4 * 7 * 4, dtype=torch.int32, device="cuda:0")
    p = C.c_void_p(buf.data_ptr())
    for limit, want in ((65536, _capi.SSD_ERR_INVALID), (65535, _capi.SSD_OK)):
        env = SSDBatchEnv("cleanup", 4, 3, map="default3", episode_limit=limit)
        before = lib.ssd_last_cuda_error()
        assert lib.ssd_set_stats(env._h, p, None) == want, limit
        assert lib.ssd_set_stats(env._h, None, p) == _capi.SSD_ERR_INVALID
        assert lib.ssd_set_stats(env._h, None, None) == _capi.SSD_OK
        assert lib.ssd_last_cuda_error() == before
        env.close()
    with pytest.raises(_capi.SsdError):
        SSDBatchEnv("cleanup", 4, 3, map="default3", episode_limit=65536, extra_args=dict(episode_stats=True))


def test_python_layer_accepts_the_option():
    import inspect
    import torch
    from homophily_marl_b200.batch_env import SSDBatchEnv
    assert "end" in inspect.signature(SSDBatchEnv.social_metrics).parameters
    assert "buf" in inspect.signature(SSDBatchEnv.stats).parameters
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            SSDBatchEnv("cleanup", 4, 3, map="default3", extra_args=dict(episode_stats=True))
