"""CPU suite: ``ssd_frontend_forward_index4`` rejects a NULL handle and NULL pointers before any CUDA call."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def test_forward_index4_rejects_null_arguments_before_any_cuda_call(lib):
    from homophily_marl_b200 import _capi
    before = lib.ssd_frontend_last_cuda_error()
    buf = C.cast((C.c_uint8 * 4096)(), C.c_void_p)
    out = C.cast((C.c_float * 4096)(), C.c_void_p)
    lut = C.cast(((C.c_uint8 * 4) * 16)(), C.c_void_p)
    fwd = lib.ssd_frontend_forward_index4
    assert fwd(None, buf, 1, 128, 8, lut, out, None) == _capi.SSD_ERR_INVALID       # V=7 strides, NULL handle
    assert fwd(None, None, 1, 128, 8, lut, out, None) == _capi.SSD_ERR_INVALID
    assert fwd(None, buf, 1, 128, 8, lut, None, None) == _capi.SSD_ERR_INVALID
    assert fwd(None, buf, 1, 128, 8, None, out, None) == _capi.SSD_ERR_INVALID
    assert fwd(None, None, 0, 0, 0, None, None, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_frontend_last_cuda_error() == before       # nothing reached the CUDA runtime
