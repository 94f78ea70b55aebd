"""GPU suite: the fused observation front end on packed colour-index observations (``ssd_frontend_forward_index4``).

The kernel only changes how a window row of pixels is loaded (two nibble words, expanded through the palette into the RGB
channel bytes), so every result must be bit-identical to ``ssd_frontend_forward`` on the RGB expansion ``lut[index]`` of the
same views: every check here is ``torch.equal`` against that, except the fp64 contract, which is restated once for V = 7,
15 and 31 so that the identity cannot hide a bug both paths share.
"""
import ctypes as C
import types

import numpy as np
import pytest

import frontend_ref as R
from obs_index_ref import obs_layout, pack, rgb_of
from test_gpu_frontend_contract import _auto_grid, _expect, _front_end, _weights

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

DEV = "cuda:0"
ROWS = 3 * 128 + 5                                            # a partial last tile


def _palette(seed):
    """16 distinct RGB entries, entry 0 non-zero: a wrong nibble or a lost bit 3 changes the bytes the conv sees."""
    rs = np.random.RandomState(seed)
    while True:
        lut = rs.randint(0, 256, size=(16, 3)).astype(np.uint8)
        if len({tuple(c) for c in lut}) == 16 and lut[0].any():
            return lut


def _indices(rows, view, seed):
    N = 2 * view + 1
    return np.random.RandomState(seed).randint(0, 16, size=(rows, N, N)).astype(np.uint8)


def _rgb_buf(lut, idx, view):
    """RGB planes lut[idx] in the env's own RGB strides (pads zero): flat u8 [rows * AS] and the layout."""
    rows, N = idx.shape[0], 2 * view + 1
    lay = R.env_layout(view)
    buf = np.zeros((rows, lay["AS"]), dtype=np.uint8)
    planes = np.lib.stride_tricks.as_strided(buf, (rows, 3, N, N), (lay["AS"], lay["PS"], lay["RP"], 1))
    planes[...] = rgb_of(lut, idx)
    return buf.reshape(-1), lay


def _packed(idx, RS=None, AS=None, garbage_seed=None):
    """index4 bytes of idx [rows, N, N] with row stride RS and agent stride AS (default: the env's); with garbage_seed every
    byte and nibble the kernel must not look at (pad nibble, row pad bytes, agent-block tail) is random instead of 0."""
    rows, N = idx.shape[0], idx.shape[-1]
    rs0, as0, _ = obs_layout(N, 1)
    RS, AS = RS or rs0, AS or as0
    if RS == rs0 and AS == as0 and garbage_seed is None:
        return pack(idx[:, None])                            # the format's own packer: [rows * agent_stride]
    buf = np.zeros((rows, AS), dtype=np.uint8) if garbage_seed is None else \
        np.random.RandomState(garbage_seed).randint(0, 256, size=(rows, AS)).astype(np.uint8)
    rows_view = np.lib.stride_tricks.as_strided(buf, (rows, N, RS), (AS, RS, 1))
    pairs = np.zeros((rows, N, 2 * ((N + 1) // 2)), dtype=np.uint8)
    pairs[..., :N] = idx
    lo, hi = pairs[..., 0::2], pairs[..., 1::2]
    if garbage_seed is not None:                              # N is odd: the high nibble of the last pixel byte is a pad
        hi[..., -1] = rows_view[..., (N - 1) // 2] >> 4
    rows_view[..., :(N + 1) // 2] = lo | (hi << 4)
    return buf.reshape(-1)


def _dev(a):
    return torch.as_tensor(a).to(DEV)


def _both(fe, lut, idx, view, RS=None, AS=None, garbage_seed=None, offset=0):
    """(RGB forward on lut[idx], index4 forward on the packed indices), synchronised."""
    rgb, lay = _rgb_buf(lut, idx, view)
    N = 2 * view + 1
    rs0, as0, _ = obs_layout(N, 1)
    packed = _packed(idx, RS, AS, garbage_seed)
    if offset:
        packed = np.concatenate([np.full(offset, 0xA5, np.uint8), packed])
    pbuf = _dev(packed)
    want = fe.forward(_dev(rgb), idx.shape[0], lay["AS"], lay["PS"], lay["RP"])
    got = fe.forward_index4(pbuf[offset:] if offset else pbuf, idx.shape[0], AS or as0, RS or rs0, lut)
    torch.cuda.synchronize()
    return want, got


# ---------------------------------------------------------------------------------------------------- identity with RGB

@pytest.mark.parametrize("view", range(1, 32))
def test_every_view_equals_the_rgb_path_bit_for_bit(view):
    lut, idx = _palette(view), _indices(ROWS, view, seed=view)
    fe = _front_end(_weights(view, seed=view), view)
    want, got = _both(fe, lut, idx, view)
    assert torch.equal(got, want), view
    assert bool(torch.isfinite(got).all())
    fe.close()


def test_a_4_column_palette_is_the_rgb0_rows_of_ssd_config():
    view = 7
    lut, idx = _palette(21), _indices(ROWS, view, seed=22)
    rgb0 = np.concatenate([lut, np.random.RandomState(23).randint(0, 256, size=(16, 1)).astype(np.uint8)], axis=1)
    fe = _front_end(_weights(view, seed=24), view)
    want, _ = _both(fe, lut, idx, view)
    got = fe.forward_index4(_dev(_packed(idx)), ROWS, obs_layout(15, 1)[1], obs_layout(15, 1)[0], torch.as_tensor(rgb0))
    assert torch.equal(got, want)                             # the 4th byte is ignored; a torch tensor palette works too
    fe.close()


@pytest.mark.parametrize("view", [7, 15, 31])
def test_fp64_contract_on_the_expansion(view):
    lut, idx = _palette(100 + view), _indices(ROWS, view, seed=200 + view)
    w = _weights(view, seed=300 + view)
    fe = _front_end(w, view)
    rgb, lay = _rgb_buf(lut, idx, view)
    rs, AS, _ = obs_layout(2 * view + 1, 1)
    got = fe.forward_index4(_dev(_packed(idx)), ROWS, AS, rs, lut)
    _expect("index4", view, got.cpu().numpy(), rgb, ROWS, lay, w, 0.01)
    fe.close()


def _env(name, mp, n, view, fmt, color, T, B=64):
    from homophily_marl_b200.batch_env import SSDBatchEnv
    extra = dict(obs_color=color, random_spawn_point=True, random_spawn_rotation=None, tag_timeout=T, obs_format=fmt,
                 disable_fire_action=False, disable_rotation_action=False)
    return SSDBatchEnv(name, B, n, map=mp, view_size=view, episode_limit=1000, extra_args=extra, seed=9, want_state=True)


@pytest.mark.parametrize("T", [0, 3])
@pytest.mark.parametrize("color", ["simplified", "full"])
@pytest.mark.parametrize("name,mp,n,view", [("cleanup", "default5", 5, 7), ("harvest", "default5", 5, 15)])
def test_env_observations_of_twin_envs(name, mp, n, view, color, T):
    """An RGB env and an index4 env stepped from one seed: the front end gives the same bits on each, out-of-play views too."""
    a, b = _env(name, mp, n, view, "rgb", color, T), _env(name, mp, n, view, "index4", color, T)
    fe = _front_end(_weights(view, seed=400 + view), view)
    a.reset()
    b.reset()
    rs = np.random.RandomState(5)
    out_seen = 0
    for t in range(30):
        act = rs.randint(0, a.n_actions, size=(a.B, a.n))
        act = np.where(rs.rand(a.B, a.n) < 0.35, 7, act).astype(np.uint8)           # FIRE often, so that agents get tagged
        at = torch.as_tensor(act, device=a.device)
        a.step(at, want_state=True)
        b.step(at, want_state=True)
        if t % 3 == 2:
            want, got = fe.forward_env(a), fe.forward_env_index4(b)
            torch.cuda.synchronize()
            assert torch.equal(got, want), t
            out_seen += int((b.tag_out > 0).sum())
    assert T == 0 or out_seen > 0
    if color == "full":
        assert int(b.obs_index().max()) >= 8                  # agent colours 8..15 were in the views
    fe.close()
    a.close()
    b.close()


# ---------------------------------------------------------------------------------------------------- bytes it must not read

@pytest.mark.parametrize("view", [3, 7, 15])
def test_pads_tails_and_other_rows_do_not_reach_a_rows_output(view):
    lut, idx = _palette(500 + view), _indices(ROWS, view, seed=600 + view)
    fe = _front_end(_weights(view, seed=700 + view), view)
    want, clean = _both(fe, lut, idx, view)
    assert torch.equal(clean, want)
    _, dirty = _both(fe, lut, idx, view, garbage_seed=1)     # pad nibble, row pad bytes and agent-block tail all random
    assert torch.equal(dirty, want)
    other = idx.copy()
    other[1::2] = _indices(ROWS, view, seed=800 + view)[1::2]
    _, got = _both(fe, lut, other, view)
    assert torch.equal(got[0::2], want[0::2])
    assert not torch.equal(got[1::2], want[1::2])
    fe.close()


def test_out_rows_beyond_rows_stay_untouched():
    view = 15
    lut, idx = _palette(31), _indices(ROWS, view, seed=32)
    fe = _front_end(_weights(view, seed=33), view)
    want, _ = _both(fe, lut, idx, view)
    rs, AS, _ = obs_layout(31, 1)
    big = torch.full((ROWS + 8, 32), float("nan"), device=DEV)
    got = fe.forward_index4(_dev(_packed(idx)), ROWS, AS, rs, lut, out=big[:ROWS])
    torch.cuda.synchronize()
    assert got.data_ptr() == big.data_ptr()
    assert torch.isnan(big[ROWS:]).all() and torch.equal(big[:ROWS], want)
    fe.close()


@pytest.mark.parametrize("view", [7, 9, 15])
@pytest.mark.parametrize("kind", ["rs+4", "rs+60", "as+4", "as+64", "offset4"])
def test_strides_beyond_the_envs(view, kind):
    N = 2 * view + 1
    rs0, as0, _ = obs_layout(N, 1)
    RS = rs0 + int(kind[3:]) if kind.startswith("rs") else rs0
    AS = {"rs": N * RS, "as": as0 + (int(kind[3:]) if kind.startswith("as") else 0)}.get(kind[:2], as0)
    lut, idx = _palette(900 + view), _indices(ROWS, view, seed=1000 + view)
    fe = _front_end(_weights(view, seed=1100 + view), view)
    want, got = _both(fe, lut, idx, view, RS=RS, AS=AS, garbage_seed=2, offset=4 if kind == "offset4" else 0)
    assert torch.equal(got, want), kind
    fe.close()


# ---------------------------------------------------------------------------------------------------- argument validation

def test_forward_index4_rejects_bad_arguments_without_a_launch():
    from homophily_marl_b200 import _capi
    view, rows = 7, 130
    N = 15
    rs, AS, _ = obs_layout(N, 1)                              # 8, 128
    fe = _front_end(_weights(view, seed=34), view)
    lib = fe.lib
    lut = np.zeros((16, 4), dtype=np.uint8)
    lut[:, :3] = _palette(35)
    buf = torch.zeros(rows * AS + 64, dtype=torch.uint8, device=DEV)
    out = torch.full((rows + 4, 32), float("nan"), device=DEV)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    before = lib.ssd_frontend_last_cuda_error()
    good_lut = lut.ctypes.data

    def fwd(obs_ptr=None, n=rows, AS=AS, RS=rs, out_ptr=None, h=fe._h):
        return lib.ssd_frontend_forward_index4(h, obs_ptr or buf.data_ptr(), n, AS, RS, good_lut, out_ptr or out.data_ptr(), stream)

    bad = [dict(RS=4), dict(RS=0), dict(RS=rs + 2), dict(RS=rs + 1), dict(AS=N * rs - 4), dict(AS=N * rs + 2), dict(AS=0),
           dict(obs_ptr=buf.data_ptr() + 1), dict(obs_ptr=buf.data_ptr() + 2), dict(out_ptr=out.data_ptr() + 4),
           dict(out_ptr=out.data_ptr() + 8), dict(n=-1), dict(h=None)]
    for kw in bad:
        assert fwd(**kw) == _capi.SSD_ERR_INVALID, kw
    assert lib.ssd_frontend_forward_index4(fe._h, buf.data_ptr(), rows, AS, rs, None, out.data_ptr(), stream) == _capi.SSD_ERR_INVALID
    assert lib.ssd_frontend_forward_index4(fe._h, None, rows, AS, rs, good_lut, out.data_ptr(), stream) == _capi.SSD_ERR_INVALID
    assert lib.ssd_frontend_forward_index4(fe._h, buf.data_ptr(), rows, AS, rs, good_lut, None, stream) == _capi.SSD_ERR_INVALID
    assert fwd(n=0, RS=4) == _capi.SSD_ERR_INVALID            # strides are checked even when there is nothing to do
    w31 = _weights(31, seed=36)
    fe31 = _front_end(w31, 31)
    tiles = (1 << 31) // 244 + 1                              # V=31: 244 chunks per tile, units = tiles * 244 >= 2^31
    rs31, as31, _ = obs_layout(63, 1)
    assert fwd(n=tiles * 128, AS=as31, RS=rs31, h=fe31._h) == _capi.SSD_ERR_INVALID
    assert fwd(n=0) == _capi.SSD_OK                           # nothing to launch
    torch.cuda.synchronize()
    assert torch.isnan(out).all()                             # nothing was launched
    assert lib.ssd_frontend_last_cuda_error() == before
    assert fwd() == _capi.SSD_OK                              # the same arguments with good strides do launch
    torch.cuda.synchronize()
    assert not torch.isnan(out[:rows]).any() and torch.isnan(out[rows:]).all()
    empty = fe.forward_index4(buf, 0, AS, rs, lut)
    assert empty.shape == (0, 32) and empty.dtype == torch.float32 and empty.is_cuda
    fe31.close()
    fe.close()


def test_forward_index4_rejects_what_forward_rejects_in_python():
    view, rows = 7, 130
    rs, AS, _ = obs_layout(15, 1)
    fe = _front_end(_weights(view, seed=37), view)
    lut = _palette(38)
    buf = torch.zeros(rows * AS, dtype=torch.uint8, device=DEV)
    bad_out = [torch.empty((rows, 32), dtype=torch.float16, device=DEV), torch.empty((rows, 31), device=DEV),
               torch.empty((rows - 1, 32), device=DEV), torch.empty((rows * 32,), device=DEV),
               torch.empty((32, rows), device=DEV).t(), torch.empty((rows, 64), device=DEV)[:, :32], torch.empty((rows, 32))]
    for out in bad_out:
        with pytest.raises(ValueError):
            fe.forward_index4(buf, rows, AS, rs, lut, out=out)
    for obs in (buf.cpu(), buf.float(), buf[:-1], torch.zeros((rows, 2 * AS), dtype=torch.uint8, device=DEV)[:, ::2]):
        with pytest.raises(ValueError):
            fe.forward_index4(obs, rows, AS, rs, lut)
    for bad_lut in (lut[:15], lut.astype(np.int32), np.zeros((16, 5), np.uint8), lut[:, :2]):
        with pytest.raises(ValueError):
            fe.forward_index4(buf, rows, AS, rs, bad_lut)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            fe.forward_index4(buf.to("cuda:1"), rows, AS, rs, lut)
        with pytest.raises(ValueError):
            fe.forward_index4(buf, rows, AS, rs, lut, out=torch.empty((rows, 32), device="cuda:1"))
    fe.close()


def test_forward_env_index4_needs_an_index4_env_and_forward_env_still_refuses_one():
    view = 7
    a, b = _env("cleanup", "default5", 5, view, "rgb", "full", 0, B=4), _env("cleanup", "default5", 5, view, "index4", "full", 0, B=4)
    fe = _front_end(_weights(view, seed=39), view)
    with pytest.raises(ValueError):
        fe.forward_env_index4(a)
    with pytest.raises(ValueError):
        fe.forward_env(b)
    fe.close()
    a.close()
    b.close()


# ---------------------------------------------------------------------------------------------------- work division

@pytest.mark.parametrize("view,rows", [(7, 2560), (15, 300), (31, 200), (3, 200)])
def test_every_grid_equals_the_rgb_path_at_that_grid(view, rows, monkeypatch):
    lut, idx = _palette(1200 + view), _indices(rows, view, seed=1300 + view)
    fe = _front_end(_weights(view, seed=1400 + view), view)
    auto, units = _auto_grid(view, rows)
    for g in [1, 2, 3, 7, 13, 64, None] + ([units] if units <= auto else []):
        if g is None:
            monkeypatch.delenv("SSD_B200_FRONTEND_GRID", raising=False)
        else:
            monkeypatch.setenv("SSD_B200_FRONTEND_GRID", str(g))
        want, got = _both(fe, lut, idx, view)
        assert torch.equal(got, want), g
    fe.close()


def test_one_handle_alternating_formats_over_growing_batches(monkeypatch):
    """131 200 rows (1 025 tiles) re-allocate the tile counters, here in an index4 call; every call must find the counters
    and scratch that the other format's calls used left clean."""
    view = 3
    fe = _front_end(_weights(view, seed=40), view)
    lut = _palette(41)
    rs, AS, _ = obs_layout(7, 1)
    seq = [(300, "1"), (300, None), (20480, "64"), (20480, None), (131200, "97"), (131200, None), (300, "7"), (20480, "2")]
    for i, (rows, grid) in enumerate(seq):
        if grid is None:
            monkeypatch.delenv("SSD_B200_FRONTEND_GRID", raising=False)
        else:
            monkeypatch.setenv("SSD_B200_FRONTEND_GRID", grid)
        idx = _indices(rows, view, seed=1500 + i)
        rgb, lay = _rgb_buf(lut, idx, view)
        packed = _dev(_packed(idx))
        if i % 2 == 0:                                        # the growing calls alternate: RGB first, then index4 first
            got = fe.forward_index4(packed, rows, AS, rs, lut)
            want = fe.forward(_dev(rgb), rows, lay["AS"], lay["PS"], lay["RP"])
        else:
            want = fe.forward(_dev(rgb), rows, lay["AS"], lay["PS"], lay["RP"])
            got = fe.forward_index4(packed, rows, AS, rs, lut)
        torch.cuda.synchronize()
        assert torch.equal(got, want), (i, rows, grid)
    fe.close()


def test_two_handles_on_two_streams_without_a_host_sync():
    view, rows = 7, 2560
    lut = _palette(42)
    rs, AS, _ = obs_layout(15, 1)
    idxs = [_indices(rows, view, seed=1600 + i) for i in range(2)]
    fes = [_front_end(_weights(view, seed=43 + i), view) for i in range(2)]
    wants = [_both(fe, lut, idx, view)[0] for fe, idx in zip(fes, idxs)]
    bufs = [_dev(_packed(idx)) for idx in idxs]
    outs = [torch.empty((rows, 32), device=DEV) for _ in range(2)]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=DEV) for _ in range(2)]
    for fe, buf, out, s in zip(fes, bufs, outs, streams):
        with torch.cuda.stream(s):
            fe.forward_index4(buf, rows, AS, rs, lut, out=out)
    torch.cuda.synchronize()
    for i in range(2):
        assert torch.equal(outs[i], wants[i]), i
    for fe in fes:
        fe.close()


# ---------------------------------------------------------------------------------------------------- batched runner

def _index4_runner(fused, obs_format="index4", B=128, T=20, G=4):
    from homophily_marl_b200.batched_runner import BatchedEpisodeRunner
    n, view = 3, 7
    extra = dict(random_spawn_point=True, random_spawn_rotation=None, disable_rotation_action=False,
                 disable_fire_action=False, obs_color="full", tag_timeout=2, obs_format=obs_format)
    env_args = dict(num_agents=n, render=False, episode_limit=T, is_replay=False, view_size=view, map="default3", extra_args=extra, seed=5)
    args = types.SimpleNamespace(batch_size_run=B, env="cleanup", env_args=env_args, device=DEV, name="homophily", mac="homophily_mac",
                                 n_actions=None, ind_reward=True, runner_log_interval=10 ** 9, test_nepisode=B, env_groups=G,
                                 fused_frontend=fused, rgb_input=True)
    return BatchedEpisodeRunner(args, types.SimpleNamespace(log_stat=lambda k, v, t: None))


def _mac(module, N, n, table, table_inc):
    class Agent:
        conv_to_fc = module

        def rgb_preprocess(self, x):
            return module(x)

    class MAC:                                                # scripted actions; the features go through rgb_preprocess
        agent = Agent()

        def init_hidden(self, batch_size):
            pass

        def select_actions_env(self, batch, t_ep, t_env, test_mode=False):
            feats = self.agent.rgb_preprocess(batch["obs"][:, t_ep].reshape(-1, 3, N, N))
            assert feats.shape == (batch.batch_size * n, 32)
            return table[batch.offset:batch.offset + batch.batch_size, t_ep].clone()

        def select_actions_inc(self, actions, batch, t_ep, t_env, test_mode=False, agent_pos_replay=None):
            return table_inc[batch.offset:batch.offset + batch.batch_size, t_ep].clone()
    return MAC()


def test_batched_runner_setup_selects_the_front_end_by_format():
    from homophily_marl_b200.frontend import MacFrontEnd
    torch.manual_seed(0)
    module = torch.nn.Sequential(torch.nn.Conv2d(3, 6, 3, 1), torch.nn.LeakyReLU(), torch.nn.Flatten(),
                                 torch.nn.Linear(6 * 13 * 13, 32), torch.nn.LeakyReLU()).to(DEV)
    mac = _mac(module, 15, 3, None, None)
    factory = dict(batch_cls=lambda *a, **k: None)
    runner = _index4_runner("index4", B=8, G=1)
    runner.setup(None, None, None, mac, **factory)
    assert isinstance(runner.front, MacFrontEnd) and runner.front.obs_format == "index4"
    runner.front.detach()
    for bad in ("rgb", "yes", 1, "INDEX4"):
        runner.args.fused_frontend = bad
        with pytest.raises(ValueError):
            runner.setup(None, None, None, mac, **factory)
    runner.close_env()
    rgb = _index4_runner("index4", obs_format="rgb", B=8, G=1)
    with pytest.raises(ValueError, match="index4"):
        rgb.setup(None, None, None, mac, **factory)
    rgb.args.fused_frontend = True
    rgb.setup(None, None, None, mac, **factory)
    assert rgb.front.obs_format == "rgb"
    rgb.front.detach()
    rgb.close_env()


def test_batched_runner_ranges_read_index4_bit_identical_to_rgb(monkeypatch):
    """env_groups = 4, index4 env, fused front end on index4: each fused call equals, bit for bit, the RGB front end (same
    handle) on the fp32 observations the runner stored for that step."""
    from homophily_marl_b200.frontend import MacFrontEnd, ObsFrontEnd
    from test_batched_runner import FakeBatch, _scheme
    B, T, n, view, G = 128, 20, 3, 7, 4
    N = 2 * view + 1
    runner = _index4_runner("index4", B=B, T=T, G=G)
    info = runner.get_env_info()
    A = runner.args.n_actions = info["n_actions"]
    g = torch.Generator().manual_seed(3)
    table = torch.randint(0, A, (B, T + 1, n, 1), generator=g).to(DEV)
    table_inc = torch.randint(0, 3, (B, T + 1, n, n, 1), generator=g).to(DEV)
    runner.use_batch_factory(lambda: FakeBatch(_scheme(n, A, *info["state_dims"], N), B, T + 1, DEV))
    torch.manual_seed(19)
    P = 2 * view - 1
    module = torch.nn.Sequential(torch.nn.Conv2d(3, 6, 3, 1), torch.nn.LeakyReLU(), torch.nn.Flatten(),
                                 torch.nn.Linear(6 * P * P, 32), torch.nn.LeakyReLU()).to(DEV)
    records = []
    forward_index4 = ObsFrontEnd.forward_index4

    def recording(self, obs_buf, rows, agent_stride, row_stride, color_lut, out=None):
        got = forward_index4(self, obs_buf, rows, agent_stride, row_stride, color_lut, out=out)
        records.append((self, got.clone(), rows))
        return got

    monkeypatch.setattr(ObsFrontEnd, "forward_index4", recording)
    runner.mac = _mac(module, N, n, table, table_inc)
    runner.front = MacFrontEnd(runner.mac, runner.env, obs_format="index4")
    batch = runner.run(test_mode=True)
    torch.cuda.synchronize()
    assert len(records) == (T + 1) * G                        # t-major, range-minor
    Bg = B // G
    lay = R.env_layout(view)
    for i, (fe, got, rows) in enumerate(records):
        t, k = divmod(i, G)
        assert rows == Bg * n
        u8 = (batch["obs"][k * Bg:(k + 1) * Bg, t] * 256).to(torch.uint8).reshape(rows, 3, N, N)
        rgb = torch.zeros((rows, lay["AS"]), dtype=torch.uint8, device=DEV)
        rgb.as_strided((rows, 3, N, N), (lay["AS"], lay["PS"], lay["RP"], 1)).copy_(u8)
        want = fe.forward(rgb.view(-1), rows, lay["AS"], lay["PS"], lay["RP"])
        assert torch.equal(got, want), (t, k)
    handles = [{id(rec[0]) for rec in records[k::G]} for k in range(G)]
    assert all(len(h) == 1 for h in handles) and len(set.union(*handles)) == G
    runner.env.set_obs_format("rgb")                          # the front end was built for index4: it must not read RGB bytes
    runner.front.active, runner.front.rows = True, (0, Bg * n)
    with pytest.raises(ValueError, match="index4"):
        runner.front(torch.zeros((Bg * n, 3, N, N), device=DEV))
    runner.front.detach()
    runner.close_env()


def test_refloop_components_with_index4_and_the_fused_front_end():
    """As test_train_loop.py::test_batched_runner_with_fused_front_end_and_device_selector, on index4 observations."""
    from baseline import refloop
    if not refloop.available():
        pytest.skip("reference sources absent (baseline/_ref)")
    from test_train_loop import _cfg
    B = 128
    env_args = dict(num_agents=3, map="default3", episode_limit=20, extra_args=dict(obs_format="index4"))
    cfg = _cfg(runner="batched", batch_size_run=B, buffer_size=2 * B, batch_size=8, buffer_cpu_only=False, fused_frontend="index4",
               action_selector="epsilon_greedy_b200", test_nepisode=B, env_args=env_args)
    c = refloop.build_components(cfg, backend="b200")
    from homophily_marl_b200.frontend import MacFrontEnd
    assert isinstance(c.runner.front, MacFrontEnd) and c.runner.front.obs_format == "index4"
    assert c.runner.env.obs_format == "index4"
    calls = {"fused": 0}
    fe = c.runner.front._front_end()
    fwd = fe.forward_index4

    def counting(*a, **k):
        calls["fused"] += 1
        return fwd(*a, **k)
    fe.forward_index4 = counting
    batch = c.runner.run(test_mode=False)
    assert calls["fused"] == 21 and bool(batch["filled"].all())               # one per select_actions_env call (T + 1)
    c.buffer.insert_episode_batch(batch)
    sample = c.buffer.sample(8)
    c.learner.train(sample[:, :sample.max_t_filled()], c.runner.t_env, B)      # optimiser step -> parameter versions change
    stamp = c.runner.front._stamp
    c.runner.run(test_mode=True)
    assert c.runner.front._stamp != stamp                                      # the weights were re-packed after the update
    c.runner.close_env()
    rgb_cfg = _cfg(runner="batched", batch_size_run=8, buffer_size=16, batch_size=8, buffer_cpu_only=False, fused_frontend="index4",
                   action_selector="epsilon_greedy_b200", test_nepisode=8, env_args=dict(num_agents=3, map="default3", episode_limit=20))
    with pytest.raises(ValueError, match="index4"):
        refloop.build_components(rgb_cfg, backend="b200")
