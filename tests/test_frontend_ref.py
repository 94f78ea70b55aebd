"""CPU suite for the fused observation front end: the float64 restatement in ``frontend_ref.py`` equals the reference module
``nn.Sequential(Conv2d(3,6,3), LeakyReLU, Flatten, Linear(6 P^2, 32), LeakyReLU)`` on ``obs / 256``, and
``ssd_frontend_create`` / ``ssd_frontend_forward`` reject bad arguments before any CUDA call."""
import ctypes as C

import numpy as np
import pytest

import frontend_ref as R

torch = pytest.importorskip("torch")


def _module(view, slope, seed):
    torch.manual_seed(seed)
    P = 2 * view - 1
    return torch.nn.Sequential(torch.nn.Conv2d(3, 6, 3, 1), torch.nn.LeakyReLU(slope), torch.nn.Flatten(),
                               torch.nn.Linear(6 * P * P, 32), torch.nn.LeakyReLU(slope)).double()


def _layouts(view):
    N = 2 * view + 1
    env = R.env_layout(view)
    RP = env["RP"] + 8
    odd = dict(RP=RP, PS=N * RP + 12, AS=3 * (N * RP + 12) + 4)             # not the env's strides; AS not a multiple of 16
    return [env, odd]


@pytest.mark.parametrize("view", [1, 2, 7, 9, 15, 17, 31])
@pytest.mark.parametrize("slope", [0.0, 0.01, 1.0])
def test_forward64_equals_the_reference_module_in_float64(view, slope):
    rows = 5
    mod = _module(view, slope, seed=view)
    with torch.no_grad():
        mod[0].bias -= 0.1                                    # both LeakyReLU branches in the conv
    w = [p.detach().numpy() for p in mod.parameters()]
    for lay in _layouts(view):
        rs = np.random.RandomState(view)
        buf = rs.randint(0, 256, size=rows * lay["AS"] + 64).astype(np.uint8)
        y, M = R.forward64(buf, rows, lay["AS"], lay["PS"], lay["RP"], view, *w, slope)
        x = torch.as_tensor(R.gather(buf, rows, lay["AS"], lay["PS"], lay["RP"], view)).double() / 256
        with torch.no_grad():
            want = mod(x).numpy()
        assert y.shape == (rows, 32) and M.shape == (rows, 32)
        assert np.abs(y - want).max() <= 1e-12 * (1 + np.abs(want).max()), (view, slope, lay)
        assert (M >= np.abs(y) - 1e-12).all()                 # |y| <= |z| <= M
        if slope == 1.0:                                      # the identity activation: the whole thing is affine
            assert np.abs(y - (R.features64(buf, rows, lay["AS"], lay["PS"], lay["RP"], view, w[0], w[1], slope) @ w[2].T + w[3])).max() < 1e-12


def test_gather_reads_through_the_strides():
    view, rows = 2, 3
    lay = dict(RP=12, PS=5 * 12 + 4, AS=3 * 64 + 8)
    buf = (np.arange(rows * lay["AS"]) % 251).astype(np.uint8)
    g = R.gather(buf, rows, lay["AS"], lay["PS"], lay["RP"], view)
    for r, c, y, x in [(0, 0, 0, 0), (2, 2, 4, 4), (1, 1, 3, 2)]:
        assert g[r, c, y, x] == buf[r * lay["AS"] + c * lay["PS"] + y * lay["RP"] + x]


def test_tf32_rounding_is_nearest_ties_away():
    one = np.float32(1.0)
    ulp = np.float32(2.0 ** -10)                              # tf32 keeps 10 mantissa bits
    vals = np.array([1.0, 1 + 2.0 ** -11, 1 + 2.0 ** -11 + 2.0 ** -20, 1 + 2.0 ** -12, -(1 + 2.0 ** -11)], dtype=np.float32)
    want = np.array([one, one + ulp, one + ulp, one, -(one + ulp)], dtype=np.float32)
    assert np.array_equal(R.tf32_rna(vals), want)
    x = np.random.RandomState(0).standard_normal(1000).astype(np.float32)
    h = R.tf32_rna(x)
    assert (h.view(np.uint32) & 0x1FFF == 0).all() and (np.abs(x - h) <= np.abs(x) * 2.0 ** -11).all()


def test_longest_chain_restates_the_rotation():
    # V: chain, from rotation() in csrc/frontend_b200.cu (min(7, ceil(steps / 24)) accumulators per issuer)
    assert {v: R.longest_chain(v) for v in (1, 7, 15, 17, 23, 31)} == {1: 6, 7: 20, 15: 50, 17: 85, 23: 116, 31: 210}
    assert all(R.tolerance(v) == 1e-6 for v in range(1, 16)) and R.tolerance(31) == pytest.approx(4.2e-6)
    assert all(R.tolerance(v) >= 1e-6 for v in range(1, 32))


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def test_frontend_create_and_forward_reject_bad_arguments_before_any_cuda_call(lib):
    from homophily_marl_b200 import _capi
    before = lib.ssd_frontend_last_cuda_error()
    view = 3
    P = 2 * view - 1
    conv_w, conv_b = np.zeros(6 * 27, np.float32), np.zeros(6, np.float32)
    fc_w, fc_b = np.zeros(32 * 6 * P * P, np.float32), np.zeros(32, np.float32)
    ptrs = [a.ctypes.data for a in (conv_w, conv_b, fc_w, fc_b)]

    def create(v=view, p=ptrs, slope=0.01, out=True):
        h = C.c_void_p(123)
        rc = lib.ssd_frontend_create(v, *p, slope, 0, C.byref(h) if out else None)
        return rc, h

    for v in (0, 32, -1):
        rc, h = create(v=v)
        assert rc == _capi.SSD_ERR_INVALID and not h.value, v
    for s in (-0.01, 1.0001, float("nan"), float("inf")):
        rc, h = create(slope=s)
        assert rc == _capi.SSD_ERR_INVALID and not h.value, s
    for i in range(4):
        p = list(ptrs)
        p[i] = None
        rc, h = create(p=p)
        assert rc == _capi.SSD_ERR_INVALID and not h.value, i
    assert create(out=False)[0] == _capi.SSD_ERR_INVALID
    buf = (C.c_uint8 * 4096)()
    out = (C.c_float * 4096)()
    assert lib.ssd_frontend_forward(None, C.cast(buf, C.c_void_p), 1, 80, 24, 8, C.cast(out, C.c_void_p), None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_frontend_forward(None, None, 0, 0, 0, 0, None, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_frontend_destroy(None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_frontend_last_cuda_error() == before       # nothing reached the CUDA runtime
