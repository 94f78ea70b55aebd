"""CPU suite: ssd_create validates tag_timeout (an 8-bit timer in the agent record) before any CUDA call."""
import ctypes as C

import pytest

from harness import ssd_config


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


@pytest.mark.parametrize("T", [-1, 256, 1 << 20])
def test_create_rejects_out_of_range_tag_timeout(lib, T):
    from homophily_marl_b200 import _capi
    h = C.c_void_p()
    assert lib.ssd_create(C.byref(ssd_config(tag_timeout=T)), C.byref(h)) == _capi.SSD_ERR_INVALID
    assert not h.value


def test_in_range_tag_timeout_passes_validation(lib):
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("GPU present: ssd_create would succeed")
    from homophily_marl_b200 import _capi
    h = C.c_void_p()
    for T in (0, 1, 255):                                          # reaches the CUDA calls, which fail without a device
        assert lib.ssd_create(C.byref(ssd_config(tag_timeout=T)), C.byref(h)) == _capi.SSD_ERR_CUDA
