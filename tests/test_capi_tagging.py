"""CPU suite: ssd_create validates tag_timeout (an 8-bit timer in the agent record) before any CUDA call."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def _cfg(**kw):
    from homophily_marl_b200 import _capi
    rows = ["@@@@@", "@P B@", "@ P @", "@@@@@"]
    cfg = _capi.SsdConfig()
    cfg.kind, cfg.n_envs, cfg.n_agents, cfg.height, cfg.width, cfg.view = 0, 4, 1, len(rows), len(rows[0]), 7
    cfg.episode_limit, cfg.fire_cost, cfg.hit_penalty, cfg.beam_len = 10, 1, 0, 5
    cfg.ascii_map = "".join(rows).encode()
    thr = (C.c_uint32 * 8)()
    cfg.thr_apple = cfg.thr_waste = C.cast(thr, C.c_void_p)
    cfg.n_waste_lut = 1
    for k, v in kw.items():
        setattr(cfg, k, v)
    cfg._keep = thr
    return cfg


@pytest.mark.parametrize("T", [-1, 256, 1 << 20])
def test_create_rejects_out_of_range_tag_timeout(lib, T):
    from homophily_marl_b200 import _capi
    h = C.c_void_p()
    assert lib.ssd_create(C.byref(_cfg(tag_timeout=T)), C.byref(h)) == _capi.SSD_ERR_INVALID
    assert not h.value


def test_in_range_tag_timeout_passes_validation(lib):
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("GPU present: ssd_create would succeed")
    from homophily_marl_b200 import _capi
    h = C.c_void_p()
    for T in (0, 1, 255):                                          # reaches the CUDA calls, which fail without a device
        assert lib.ssd_create(C.byref(_cfg(tag_timeout=T)), C.byref(h)) == _capi.SSD_ERR_CUDA
