"""CPU suite: ``ssd_set_view_offset`` (DESIGN.md §3 item 18) is exported and declared, and refuses a NULL handle with
SSD_ERR_INVALID before any CUDA call, whatever the offset."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def test_symbol_is_exported_and_declared(lib):
    from homophily_marl_b200 import _capi
    assert hasattr(lib, "ssd_set_view_offset") and "ssd_set_view_offset" in _capi.EXPORTS
    text = open(os.path.join(ROOT, "include", "ssd_b200.h")).read()
    assert re.search(r"int ssd_set_view_offset\(ssd_handle\* h, int32_t offset\);", text)
    assert lib.ssd_abi_version() == 2


def test_null_handle_is_refused_before_any_cuda_call(lib):
    from homophily_marl_b200 import _capi
    before = lib.ssd_last_cuda_error()
    for offset in (0, 1, 15, 31, -1, 32, 2 ** 31 - 1, -2 ** 31):
        assert lib.ssd_set_view_offset(None, C.c_int32(offset)) == _capi.SSD_ERR_INVALID, offset
    assert lib.ssd_last_cuda_error() == before
