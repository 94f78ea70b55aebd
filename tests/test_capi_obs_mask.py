"""CPU suite: the row-mask calls of the C ABI (ssd_obs_mask_words, ssd_set_obs_mask; DESIGN.md §3 item 19) refuse a NULL handle
before any CUDA call, and the Python binding declares them."""
import pytest


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def test_null_handle_is_refused(lib):
    from homophily_marl_b200 import _capi
    assert "ssd_obs_mask_words" in _capi.EXPORTS and "ssd_set_obs_mask" in _capi.EXPORTS
    assert lib.ssd_obs_mask_words(None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_set_obs_mask(None, None, None, None, None) == _capi.SSD_ERR_INVALID
